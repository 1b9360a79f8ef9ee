// kernels.cuh -- the sm_100a kernels of the slot-commitment path (K1..K6 of SURVEY.md section 2).
//
// HBM layout: every retained Merkle layer is a dense array of canonical 32-byte little-endian field elements
// (what crosses the C ABI), so sampled paths are plain gathers.  Inside a kernel the state is Montgomery-form
// 8x32-bit limbs in registers; conversion happens at the load/store edge (3 extra modmuls per 240-modmul
// permutation at most).
//
// None of these kernels is HBM-bound: one cell is 2048 B in, 32 B out and 34*240 = 8160 modmuls = 1.1 M
// integer-multiply instructions.  The bound is the FMA-pipe IMAD.WIDE issue rate (DESIGN.md, "Roofline").
#pragma once
#include "poseidon2.cuh"

namespace cdx {

static __device__ __forceinline__ Fr ld_felt(const uint8_t* p) {   // p is 16-byte aligned
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  Fr r = {{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
  return r;
}

static __device__ __forceinline__ void st_felt(uint8_t* p, const Fr& v) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
  q[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

#ifndef CDX_BLOCK
#define CDX_BLOCK 256
#endif

// first statement of every kernel that does field arithmetic: the CTA's copy of the reduction table (fr.cuh), before any
// thread can leave
#if CDX_TABRED
#define CDX_KERNEL_PROLOGUE() load_reduce_tab()
#else
#define CDX_KERNEL_PROLOGUE() ((void)0)
#endif

// K1: n independent permutations (BASELINE config 2).           Permutation.hs:40-45
__global__ void __launch_bounds__(CDX_BLOCK) k_permutation_batch(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, size_t n) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr x = to_mont(ld_felt(in + 96 * i)), y = to_mont(ld_felt(in + 96 * i + 32)), z = to_mont(ld_felt(in + 96 * i + 64));
  permute(x, y, z);
  st_felt(out + 96 * i, from_mont(x));
  st_felt(out + 96 * i + 32, from_mont(y));
  st_felt(out + 96 * i + 64, from_mont(z));
}

// sponge over field elements, one sponge per thread.             Sponge.hs:13-43
__global__ void __launch_bounds__(CDX_BLOCK) k_sponge_felts(const uint8_t* __restrict__ elems, size_t n_items, uint32_t len, int rate,
                                                            uint8_t* __restrict__ out) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items) return;
  const uint8_t* base = elems + (size_t)32 * len * i;
  auto get = [&](uint32_t k) { return ld_felt(base + 32 * k); };
  st_felt(out + 32 * i, from_mont(sponge_elems(get, len, rate)));
}

// K2: cell sponge, one cell per thread (a warp covers 32 consecutive cells = one 64 KiB block at the default
// sizes).  Cells are 4-byte aligned and a multiple of 4 bytes long.        blocks/bn254.nim:23-29, Slot.hs:222-228
__global__ void __launch_bounds__(CDX_BLOCK) k_hash_cells(const uint32_t* __restrict__ data, size_t n_cells, uint32_t cell_words,
                                                          uint8_t* __restrict__ out) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_cells) return;
  AlignedWords ld{data + (size_t)cell_words * i, cell_words};
  st_felt(out + 32 * i, from_mont(sponge2_bytes(ld, cell_words * 4u)));
}

// K2 with TMA-staged rows.  Same arithmetic; the slot bytes reach the threads through shared memory instead of
// per-thread global loads.  The slot is described to the TMA unit as a 2-D byte tensor [n_cells][cell_bytes]; a warp
// (32 consecutive cells) fetches the next 32-byte column segment of all its cells with ONE tensor copy
// (cp.async.bulk.tensor.2d -> SASS UTMALDG) issued by one elected lane into a ring of CDX_RING_SLOTS boxes of
// 32 rows x 32 B, two segments ahead of the sponge.  One mbarrier per (warp, ring slot): expect_tx = 1024 B, the phase
// completes when the box has landed (rows past the end of the slot are zero-filled by the TMA unit and still counted).
// Lane l only ever reads row l, and a box is overwritten only after the step that last read it: begin_step opens with a
// __syncwarp(), which orders every lane's reads of step j-1 before the elected lane's refill.
//   HBM traffic: each 32-byte sector of the slot is fetched exactly once.
#ifndef CDX_RING_SLOTS
#define CDX_RING_SLOTS 6
#endif
// resident CTAs per SM the cell kernel is compiled for: 3 x 256 threads = 24 warps at 80 registers, no spills.  With the
// table-driven reduction the kernel is insensitive to occupancy (same-box sweep, profiles/r2_sweep_occupancy.txt: 16 to 32
// warps per SM within 0.2 %); this point was the fastest and leaves room for the 4 KB reduction table next to the rings.
#ifndef CDX_TMA_MIN_CTAS
#define CDX_TMA_MIN_CTAS 3
#endif
#define CDX_SEG_BYTES 32u
#define CDX_BOX_BYTES (32u * CDX_SEG_BYTES)

struct RowRing {
  // Deliberately (almost) stateless: everything is re-derived from the step number and the thread indices once per
  // step (a step is one permutation, ~45 k instructions), so nothing of the pipeline lives in registers across the
  // permutation -- the hot loops then get the same register allocation as in the plain-load kernel.
  const void* tmap;       // the slot as a 2-D tensor (kernel parameter space: no register cost)
  uint32_t smem_base;     // 128-byte aligned shared-space base of the CTA's rings
  uint32_t cell_bytes;

  __device__ __forceinline__ uint32_t warp() const { return threadIdx.x >> 5; }
  __device__ __forceinline__ uint32_t boxes() const { return smem_base + warp() * (CDX_RING_SLOTS * CDX_BOX_BYTES); }
  __device__ __forceinline__ uint32_t bars() const {
    return smem_base + (blockDim.x >> 5) * (CDX_RING_SLOTS * CDX_BOX_BYTES) + warp() * (8u * CDX_RING_SLOTS);
  }
  __device__ __forceinline__ int last_seg() const { return (int)(cell_bytes / CDX_SEG_BYTES) - 1; }
  // segments wanted resident-or-in-flight / needed landed when step j starts (-1 before the first step)
  __device__ __forceinline__ int want_at(int j) const {
    if (j < 0) return -1;
    const int w = (int)((62u * (uint32_t)j) / CDX_SEG_BYTES) + (CDX_RING_SLOTS - 1);
    return w < last_seg() ? w : last_seg();
  }
  __device__ __forceinline__ int need_at(int j) const {
    if (j < 0) return -1;
    const int h = (int)((62u * (uint32_t)j + 67u) / CDX_SEG_BYTES);
    return h < last_seg() ? h : last_seg();
  }
  // step j of the sponge reads padded-stream bytes [62 j, 62 j + 68): make those segments resident, keep two ahead
  __device__ __forceinline__ void begin_step(uint32_t j) const {
    const int issued = want_at((int)j - 1), want = want_at((int)j);
    // every lane has finished reading the boxes of step j-1 (and has passed its waits on their barriers) before the
    // elected lane re-arms a barrier and lets the async proxy overwrite a box: convergence is not assumed
    __syncwarp();
    if ((threadIdx.x & 31u) == 0) {
      const uint32_t row0 = blockIdx.x * blockDim.x + (threadIdx.x & ~31u);          // first cell (tensor row) of this warp
      for (int g = issued + 1; g <= want; ++g) {
        const uint32_t slot = (uint32_t)g % CDX_RING_SLOTS;
        const uint32_t bar = bars() + 8u * slot;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(CDX_BOX_BYTES) : "memory");
        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                         boxes() + slot * CDX_BOX_BYTES),
                     "l"(tmap), "r"((uint32_t)g * CDX_SEG_BYTES), "r"(row0), "r"(bar)
                     : "memory");
      }
    }
    __syncwarp();
    for (int g = need_at((int)j - 1) + 1; g <= need_at((int)j); ++g) {
      const uint32_t bar = bars() + 8u * ((uint32_t)g % CDX_RING_SLOTS);
      const uint32_t parity = ((uint32_t)g / CDX_RING_SLOTS) & 1u;
      uint32_t done;
      do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done)
                     : "r"(bar), "r"(parity)
                     : "memory");
      } while (!done);
    }
  }
  __device__ __forceinline__ uint32_t operator()(uint32_t i) const {
    if (i >= (cell_bytes >> 2)) return i == (cell_bytes >> 2) ? 1u : 0u;
    const uint32_t seg = i >> 3, slot = seg % CDX_RING_SLOTS;
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(boxes() + slot * CDX_BOX_BYTES + (threadIdx.x & 31u) * CDX_SEG_BYTES + 4u * (i & 7u)) : "memory");
    return v;
  }
};

struct alignas(64) TensorMap2D {   // layout-compatible with CUtensorMap (128 opaque bytes, 64-byte aligned)
  unsigned long long opaque[16];
};

// cell_bytes % 32 == 0; dynamic shared memory: 128 B slack + warps x (CDX_RING_SLOTS x 1 KiB) + barriers
__global__ void __launch_bounds__(CDX_BLOCK, CDX_TMA_MIN_CTAS) k_hash_cells_tma(const __grid_constant__ TensorMap2D tmap, size_t n_cells, uint32_t cell_bytes,
                                                              uint8_t* __restrict__ out) {
  extern __shared__ uint8_t smem[];
  CDX_KERNEL_PROLOGUE();
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, n_warps = blockDim.x >> 5;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t warp_first = i - lane;
  if (warp_first >= n_cells) return;                                   // whole warp past the end (warp-uniform)
  const uint32_t smem_base = ((uint32_t)__cvta_generic_to_shared(smem) + 127u) & ~127u;   // tensor copies need 128-byte aligned boxes
  const uint32_t bars = smem_base + n_warps * (CDX_RING_SLOTS * CDX_BOX_BYTES) + warp * (8u * CDX_RING_SLOTS);
  if (lane == 0) {
#pragma unroll
    for (uint32_t s = 0; s < CDX_RING_SLOTS; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bars + 8u * s) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncwarp();
  RowRing ld;
  ld.tmap = &tmap;
  ld.smem_base = smem_base;
  ld.cell_bytes = cell_bytes;
  const Fr h = from_mont(sponge2_bytes(ld, cell_bytes));               // lanes past the end hash zero-filled rows, store nothing
  if (i < n_cells) st_felt(out + 32 * i, h);
}

// byte strings of arbitrary length/alignment (test-vector suite: n = 0..80).   testvectors.nim:41-46
__global__ void __launch_bounds__(CDX_BLOCK) k_hash_bytes_any(const uint8_t* __restrict__ data, size_t n_items, uint32_t len,
                                                              uint8_t* __restrict__ out) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items) return;
  AnyBytes ld{data + (size_t)len * i, len};
  st_felt(out + 32 * i, from_mont(sponge2_bytes(ld, len)));
}

// keyed compression batch.                                       Merkle.hs:202-203, merkle/bn254.nim:18
__global__ void __launch_bounds__(CDX_BLOCK) k_compress_batch(const uint8_t* __restrict__ x, const uint8_t* __restrict__ y,
                                                              const uint32_t* __restrict__ keys, size_t n, uint8_t* __restrict__ out) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  st_felt(out + 32 * i, from_mont(compress_keyed(to_mont(ld_felt(x + 32 * i)), to_mont(ld_felt(y + 32 * i)), keys[i] & 3u)));
}

// The Merkle node rule: node i of the level above `in` (n nodes) = compress(in[2i], in[2i+1], bottom); a trailing single
// child is paired with 0 under key bottom+2 (merkle/bn254.nim:38-53, Merkle.hs:156-178).  singles != 0: every input is a
// one-leaf tree of its own -> node i = compress(in[i], 0, 3) (Merkle.hs:73).  Canonical standard form.
static __device__ __forceinline__ Fr merkle_node(const uint8_t* __restrict__ in, size_t n, size_t i, uint32_t bottom, int singles) {
  Fr x, y;
  uint32_t key = bottom;
  if (singles) {
    x = to_mont(ld_felt(in + 32 * i));
    y = fr_zero();
    key = 3u;
  } else {
    x = to_mont(ld_felt(in + 64 * i));
    if (2 * i + 1 < n) {
      y = to_mont(ld_felt(in + 64 * i + 32));
    } else {
      y = fr_zero();
      key = bottom + 2u;
    }
  }
  return from_mont(compress_keyed(x, y, key));
}

// K3: one Merkle level, out[i] = merkle_node(in, n, i).  The same kernel reduces the forest of block trees (their widths
// are powers of two, so pairs never straddle two blocks) and every slot/dataset level.
__global__ void __launch_bounds__(CDX_BLOCK) k_merkle_level(const uint8_t* __restrict__ in, size_t n, uint8_t* __restrict__ out,
                                                            uint32_t bottom, int singles) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t n_out = singles ? n : (n + 1) / 2;
  if (i >= n_out) return;
  st_felt(out + 32 * i, merkle_node(in, n, i, bottom, singles));
}

// ---- checking an imported slot image (cdx_slot_import) ------------------------------------------------------------------
// The retained levels of an image form one chain, bottom up: a full image's block-forest levels 0..block_depth and then slot
// levels 1..slot_depth (slot level 1 is built from the block hashes, forest level block_depth); a compact image's slot
// levels 0..slot_depth.  Every stored node above the bottom level must be what the node rule makes of its stored children,
// and every stored element must be canonical.  Both use stored values only, so one launch covers every level in place.
#define CDX_IMAGE_LEVELS 72                    // 33 block-forest levels + slot levels 1..39 (slot_image.h)

struct ImageLevel {
  const uint8_t* nodes;
  uint64_t n;                                  // nodes of this level
  uint64_t first;                              // its first thread: the prefix sum of n over the levels below
  uint8_t tree, level, bottom, singles;        // tree 0 = block forest, 1 = slot tree; node rule of the level below
};

struct ImageChain {
  ImageLevel lv[CDX_IMAGE_LEVELS];
  uint32_t n_levels;
};

static __device__ __forceinline__ bool fr_is_canonical(const Fr& a) {
  const uint32_t r[8] = {CDX_N0, CDX_N1, CDX_N2, CDX_N3, CDX_N4, CDX_N5, CDX_N6, CDX_N7};
#pragma unroll
  for (int k = 7; k >= 0; --k)
    if (a.l[k] != r[k]) return a.l[k] < r[k];
  return false;
}

// the key of a bad node: smaller is (forest before slot tree, lower level, lower node, "not canonical" before "does not hash")
static __host__ __device__ __forceinline__ unsigned long long image_bad_key(uint32_t tree, uint32_t level, uint64_t node, uint32_t hashes) {
  return ((unsigned long long)tree << 63) | ((unsigned long long)level << 57) | (node << 1) | hashes;
}

// one thread per stored node (nodes < 2^56 a level: an image's levels are allocated in HBM); bad = the smallest key
__global__ void __launch_bounds__(CDX_BLOCK) k_check_image(const __grid_constant__ ImageChain chain, uint64_t total, unsigned long long* __restrict__ bad) {
  CDX_KERNEL_PROLOGUE();
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  uint32_t lo = 0, hi = chain.n_levels;        // the level with first <= t < first + n
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (chain.lv[mid].first <= t) lo = mid;
    else hi = mid;
  }
  const ImageLevel& L = chain.lv[lo];
  const uint64_t i = t - L.first;
  const Fr v = ld_felt(L.nodes + 32 * i);
  unsigned long long key = ~0ull;
  if (!fr_is_canonical(v)) {
    key = image_bad_key(L.tree, L.level, i, 0);
  } else if (lo > 0) {
    const ImageLevel& C = chain.lv[lo - 1];
    const Fr h = merkle_node(C.nodes, C.n, i, L.bottom, L.singles);
    bool same = true;
#pragma unroll
    for (int k = 0; k < 8; ++k) same &= h.l[k] == v.l[k];
    if (!same) key = image_bad_key(L.tree, L.level, i, 1);
  }
  if (key != ~0ull) atomicMin(bad, key);
}

// elements in place to canonical standard form: any 256-bit input is taken mod r.  The bottom layer a caller hands to
// cdx_merkle_layers_host comes back as layer 0, and outputs are canonical (include/codex_commit.h).
__global__ void __launch_bounds__(CDX_BLOCK) k_canonical_felts(uint8_t* __restrict__ p, size_t n) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  st_felt(p + 32 * i, from_mont(to_mont(ld_felt(p + 32 * i))));
}

// K3b: one level of MANY Merkle trees at once -- the slot trees of a batch of small slots.  The level-l nodes of all trees
// are stored tree after tree; in_off / out_off (n_trees + 1 entries each) are the prefix sums of the per-tree widths at
// the input and the output level.  Per tree the rules are those of k_merkle_level: a trailing single child is paired
// with 0 under key bottom+2, which also gives a one-leaf tree its key-3 compression at the bottom level; a tree that
// has already reached its root has output width 0 and is skipped.  A tree's root (output width 1) is also copied to
// roots[tree].                                                      merkle/bn254.nim:29-60, gen_input/bn254.nim:41-47
__global__ void __launch_bounds__(CDX_BLOCK) k_merkle_level_seg(const uint8_t* __restrict__ in, const uint64_t* __restrict__ in_off,
                                                                uint8_t* __restrict__ out, const uint64_t* __restrict__ out_off, uint32_t n_trees,
                                                                uint32_t bottom, uint8_t* __restrict__ roots) {
  CDX_KERNEL_PROLOGUE();
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out_off[n_trees]) return;
  uint32_t lo = 0, hi = n_trees;                     // largest t with out_off[t] <= i (empty trees share their offset with the next one)
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (out_off[mid] <= i) lo = mid;
    else hi = mid;
  }
  const uint64_t j = i - out_off[lo], base = in_off[lo], n = in_off[lo + 1] - base;
  const Fr x = to_mont(ld_felt(in + 32 * (base + 2 * j)));
  Fr y = fr_zero();
  uint32_t key = bottom + 2u;
  if (2 * j + 1 < n) {
    y = to_mont(ld_felt(in + 32 * (base + 2 * j + 1)));
    key = bottom;
  }
  const Fr h = from_mont(compress_keyed(x, y, key));
  st_felt(out + 32 * i, h);
  if (out_off[lo + 1] - out_off[lo] == 1) st_felt(roots + 32 * (size_t)lo, h);
}

// Runs of `width` 32-byte elements: run i of src goes to run index[i] of dst, dst[index[i] * width + k] = src[i * width + k].
// Width 1 moves the roots of a batch of slots into their places among a dataset's slot roots; a slot builder moves each
// level of a tile's block trees (width = that level's nodes per block) into the slot's forest.  One thread per 16-byte half.
__global__ void k_scatter_felts(const uint8_t* __restrict__ src, const uint64_t* __restrict__ index, size_t n, uint8_t* __restrict__ dst,
                                uint32_t width = 1) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 2 * n * width) return;
  const size_t e = t >> 1, half = t & 1, i = e / width, k = e - i * width;
  reinterpret_cast<uint4*>(dst + 32 * (index[i] * width + k))[half] = reinterpret_cast<const uint4*>(src + 32 * e)[half];
}

// K4: batched path gather.  One thread per (sample, level, 16-byte half).  Pure data movement.
//                                                                 merkle.nim:21-42,86-100, types.nim:27-37
struct PathPlan {
  const uint8_t* forest[32];   // block-forest level l (local cells >> l nodes), l < block_depth
  const uint8_t* low[40];      // slot-tree level l for l < top_level: local nodes starting at low_first[l]
  const uint8_t* top[40];      // slot-tree level l for l >= top_level: all global nodes
  uint64_t low_first[40];
  uint64_t low_count[40];
  uint64_t width[40];          // global width of slot-tree level l
  uint64_t first_cell, n_local_cells;
  uint32_t block_depth, slot_depth, top_level, cells_per_block_log2;
  uint32_t singles;            // one-cell blocks: the block-tree sibling is out of range, i.e. zero (merkle.nim:34)
};

__global__ void k_gather_paths(PathPlan plan, const uint64_t* __restrict__ cells, uint32_t n_samples, uint32_t max_depth,
                               uint8_t* __restrict__ out, uint8_t* __restrict__ leaf_out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t per_sample = (max_depth + 1) * 2;             // +1: the leaf itself
  if (t >= n_samples * per_sample) return;
  const uint32_t s = t / per_sample, rem = t % per_sample, lvl = rem >> 1, half = rem & 1u;
  const uint64_t cell = cells[s];
  const bool mine = cell >= plan.first_cell && cell < plan.first_cell + plan.n_local_cells;
  const uint64_t lc = cell - plan.first_cell;                  // local cell index (valid if mine)
  uint4 v = make_uint4(0, 0, 0, 0);
  if (lvl == max_depth) {                                      // leaf slot
    if (leaf_out == nullptr) return;
    if (mine) v = reinterpret_cast<const uint4*>(plan.forest[0] + 32 * lc)[half];
    reinterpret_cast<uint4*>(leaf_out + 32 * (size_t)s)[half] = v;
    return;
  }
  if (mine) {
    if (lvl < plan.block_depth) {
      const uint64_t sib = (lc >> lvl) ^ 1ull;                 // block trees are full: sibling always exists
      if (!plan.singles) v = reinterpret_cast<const uint4*>(plan.forest[lvl] + 32 * sib)[half];
    } else if (lvl < plan.block_depth + plan.slot_depth) {
      const uint32_t l = lvl - plan.block_depth;
      const uint64_t node = (cell >> plan.cells_per_block_log2) >> l;
      const uint64_t sib = node ^ 1ull;
      if (sib < plan.width[l]) {                               // out of range -> zero (merkle.nim:34)
        if (l >= plan.top_level) v = reinterpret_cast<const uint4*>(plan.top[l] + 32 * sib)[half];
        else if (sib >= plan.low_first[l] && sib < plan.low_first[l] + plan.low_count[l])
          v = reinterpret_cast<const uint4*>(plan.low[l] + 32 * (sib - plan.low_first[l]))[half];
      }
    }
  }
  reinterpret_cast<uint4*>(out + 32 * ((size_t)s * max_depth + lvl))[half] = v;
}

// Verifier walk, one proof per thread: reconstructRoot (merkle.nim:51-74) == RootFromMerklePath (merkle.circom:44-114).
// paths: n x stride elements (only the first `depth` of each are walked), leaves/indices: n.
__global__ void __launch_bounds__(CDX_BLOCK) k_reconstruct_roots(const uint8_t* __restrict__ leaves, const uint64_t* __restrict__ indices,
                                                                 uint64_t n_leaves, const uint8_t* __restrict__ paths, uint32_t stride,
                                                                 uint32_t depth, size_t n, uint8_t* __restrict__ out) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t j = indices[i], m = n_leaves;
  Fr h = to_mont(ld_felt(leaves + 32 * i));
  uint32_t bottom = 1;
#pragma unroll 1
  for (uint32_t l = 0; l < depth; ++l) {
    const Fr p = to_mont(ld_felt(paths + 32 * ((size_t)i * stride + l)));
    if (j & 1) h = compress_keyed(p, h, bottom);              // odd index: the sibling is on the left
    else if (j == m - 1) h = compress_keyed(h, p, bottom + 2);   // last and even: a single child (odd node)
    else h = compress_keyed(h, p, bottom);
    bottom = 0;
    j >>= 1;
    m = (m + 1) >> 1;
  }
  st_felt(out + 32 * i, from_mont(h));
}

// K5: sampled cell indices, one thread per (challenge, counter).   sample/bn254.nim:16-27, types/bn254.nim:47-59
// entropies: n_challenges x 32 B, root: 32 B (both canonical), out[ch * n_samples + c-1].
static __device__ __forceinline__ uint64_t cell_index(const uint8_t* entropy, const uint8_t* root, uint32_t counter, uint64_t mask) {
  auto get = [&](uint32_t k) {
    if (k == 0) return ld_felt(entropy);
    if (k == 1) return ld_felt(root);
    Fr c = fr_zero();
    c.l[0] = counter;
    return c;
  };
  Fr h = from_mont(sponge_elems(get, 3, 2));
  return (((uint64_t)h.l[1] << 32) | h.l[0]) & mask;
}

__global__ void k_cell_indices(const uint8_t* __restrict__ entropies, const uint8_t* __restrict__ root, uint64_t mask, uint32_t n_samples,
                               size_t total, uint64_t* __restrict__ out) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t ch = i / n_samples;
  out[i] = cell_index(entropies + 32 * ch, root, (uint32_t)(i % n_samples) + 1u, mask);   // counters run 1..nSamples
}

// K5b: the same over challenges against different slots: challenge ch samples the slot whose root is roots[ch] and whose
// cell count is masks[ch] + 1.
__global__ void k_cell_indices_rows(const uint8_t* __restrict__ entropies, const uint8_t* const* __restrict__ roots,
                                    const uint64_t* __restrict__ masks, uint32_t n_samples, size_t total, uint64_t* __restrict__ out) {
  CDX_KERNEL_PROLOGUE();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t ch = i / n_samples;
  out[i] = cell_index(entropies + 32 * ch, roots[ch], (uint32_t)(i % n_samples) + 1u, masks[ch]);
}

// the reference's fake data for the cell with global index `cell` (cell_size % 4 == 0)
static __device__ __forceinline__ void fake_cell(uint64_t seed, uint64_t cell, uint32_t cell_size, uint32_t* __restrict__ dst) {
  const uint64_t seed1 = seed + 0xdeadcafeull, seed2 = cell + 0x98765432ull;
  uint64_t s = 1;
  for (uint32_t w = 0; w < cell_size / 4; ++w) {
    uint32_t word = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      s = s * (s + seed1) * (s + seed2) + s * (s ^ 0x5a5a5a5aull) + seed1 * s + (seed2 + 17);
      s %= 1698428844001831ull;
      word |= (uint32_t)(s & 0xff) << (8 * b);
    }
    dst[w] = word;
  }
}

// word w of a synthetic slot seeded with `seed`: splitmix64(seed + w)
static __device__ __forceinline__ uint64_t synthetic_word(uint64_t seed, uint64_t w) {
  uint64_t z = seed + w + 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

// K6a: the reference's fake data, one cell per thread.            slot.nim:23-32, Slot.hs:87-96
__global__ void k_fake_cells(uint64_t seed, uint64_t first_cell, size_t n_cells, uint32_t cell_size, uint8_t* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_cells) return;
  fake_cell(seed, first_cell + i, cell_size, reinterpret_cast<uint32_t*>(out + (size_t)cell_size * i));
}

// K6b: counter-based synthetic bytes for the large benchmark slots: word i = splitmix64(seed + first_word + i).
__global__ void k_fill_synthetic(uint64_t seed, uint64_t first_word, size_t n_words, uint64_t* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (size_t)gridDim.x * blockDim.x)
    out[i] = synthetic_word(seed, first_word + i);
}

// K6c: the same stream in 4-byte halves, for a byte range or a destination that is not 8-byte aligned: half h (h = byte / 4)
// is the low (h even) or high (h odd) 32 bits of word h / 2, i.e. the bytes of the stream in little-endian order.
__global__ void k_fill_synthetic_halves(uint64_t seed, uint64_t first_half, size_t n_halves, uint32_t* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_halves; i += (size_t)gridDim.x * blockDim.x) {
    const uint64_t h = first_half + i;
    out[i] = (uint32_t)(synthetic_word(seed, h >> 1) >> (32 * (h & 1)));
  }
}

// ---- answering challenges from compact slots (cdx_slots_prove_from_source) ----------------------------------------------
// Only the slot trees are retained; the sampled blocks' bytes are brought back, re-hashed into a "sampled forest" (the
// block trees of the unique sampled (slot, block) pairs, laid out like the block forest of a slot made of just those
// blocks), checked against the retained block hashes, and the paths are gathered from both.  Every slot of one call has
// the same geometry, so the pairs of all slots share the forest's levels.

struct SlotLevel {             // one retained slot-tree level: all global nodes of it
  const uint8_t* nodes;
  uint64_t width;
};

struct SampledSlot {           // one distinct slot of the call, in the order of its first challenge row
  uint64_t seed;               // generated sources: the slot's seed
  uint64_t first_row;          // its first challenge row (the mismatch key)
  uint32_t levels;             // its slot level 0 in the level table; levels .. levels + slot_depth
  uint32_t slot_depth;
};

// K6d: generated bytes of a LIST of (slot, block) pairs, back to back: block blocks[b] of slot slot_of[b] lands at
// out + b * block_size.  fake != 0: the reference's fake data, one cell per thread; else the synthetic stream in 4-byte
// halves (block sizes need not be multiples of 8).  Grid-stride: one launch per tile whatever the number of blocks.
__global__ void k_generate_blocks(uint32_t fake, const SampledSlot* __restrict__ slots, const uint32_t* __restrict__ slot_of,
                                  const uint64_t* __restrict__ blocks, size_t n_blocks, uint64_t block_size, uint32_t cell_size,
                                  uint8_t* __restrict__ out) {
  const uint64_t per_block = fake ? block_size / cell_size : block_size / 4;    // cells or halves
  const size_t n = n_blocks * per_block;
  for (size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x; u < n; u += (size_t)gridDim.x * blockDim.x) {
    const uint64_t b = u / per_block, k = u % per_block, g = blocks[b] * per_block + k;
    const uint64_t seed = slots[slot_of[b]].seed;
    if (fake) fake_cell(seed, g, cell_size, reinterpret_cast<uint32_t*>(out + (size_t)cell_size * u));
    else reinterpret_cast<uint32_t*>(out)[u] = (uint32_t)(synthetic_word(seed, g >> 1) >> (32 * (g & 1)));
  }
}

// the recomputed hash of sampled pair i against its slot's retained level 0; bad = the smallest key (slot's first row << 44
// | block) among the pairs that differ
__global__ void k_check_sampled_blocks(const uint8_t* __restrict__ sampled, const uint64_t* __restrict__ blocks,
                                       const uint32_t* __restrict__ slot_of, size_t n, const SampledSlot* __restrict__ slots,
                                       const SlotLevel* __restrict__ levels, unsigned long long* __restrict__ bad) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const SampledSlot& sl = slots[slot_of[i]];
  const uint4* a = reinterpret_cast<const uint4*>(sampled + 32 * i);
  const uint4* c = reinterpret_cast<const uint4*>(levels[sl.levels].nodes + 32 * blocks[i]);
  const uint4 a0 = a[0], a1 = a[1], c0 = c[0], c1 = c[1];
  if (a0.x != c0.x || a0.y != c0.y || a0.z != c0.z || a0.w != c0.w || a1.x != c1.x || a1.y != c1.y || a1.z != c1.z || a1.w != c1.w)
    atomicMin(bad, (unsigned long long)((sl.first_row << 44) | blocks[i]));
}

struct SampledPathPlan {
  const uint8_t* forest[32];   // sampled-forest level l, l < block_depth
  const uint32_t* row_slot;    // challenge row -> its slot record
  const SampledSlot* slots;
  const SlotLevel* levels;
  uint32_t block_depth, cells_per_block_log2, n_samples;
  uint32_t singles;            // one-cell blocks: the block-tree sibling is out of range, i.e. zero (merkle.nim:34)
};

// K4 for compact slots: per row, the output of k_gather_paths on that row's slot over the same indices.  pos[s] is the
// position of sample s's (slot, block) pair in the sampled forest; sample s belongs to row s / n_samples.  A slot shallower
// than max_depth gets zeros above its slot depth.  One thread per (sample, level, 16-byte half).
__global__ void k_gather_paths_sampled(SampledPathPlan plan, const uint64_t* __restrict__ cells, const uint32_t* __restrict__ pos,
                                       uint32_t n_samples, uint32_t max_depth, uint8_t* __restrict__ out, uint8_t* __restrict__ leaf_out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t per_sample = (max_depth + 1) * 2;             // +1: the leaf itself
  if (t >= n_samples * per_sample) return;
  const uint32_t s = t / per_sample, rem = t % per_sample, lvl = rem >> 1, half = rem & 1u;
  const uint64_t cell = cells[s];
  const uint64_t lc = ((uint64_t)pos[s] << plan.cells_per_block_log2) | (cell & ((1ull << plan.cells_per_block_log2) - 1));   // in the sampled forest
  uint4 v = make_uint4(0, 0, 0, 0);
  if (lvl == max_depth) {                                      // leaf slot
    reinterpret_cast<uint4*>(leaf_out + 32 * (size_t)s)[half] = reinterpret_cast<const uint4*>(plan.forest[0] + 32 * lc)[half];
    return;
  }
  if (lvl < plan.block_depth) {
    if (!plan.singles) v = reinterpret_cast<const uint4*>(plan.forest[lvl] + 32 * ((lc >> lvl) ^ 1ull))[half];
  } else {
    const SampledSlot& sl = plan.slots[plan.row_slot[s / plan.n_samples]];
    const uint32_t l = lvl - plan.block_depth;
    if (l < sl.slot_depth) {
      const SlotLevel lv = plan.levels[sl.levels + l];
      const uint64_t sib = ((cell >> plan.cells_per_block_log2) >> l) ^ 1ull;
      if (sib < lv.width) v = reinterpret_cast<const uint4*>(lv.nodes + 32 * sib)[half];   // out of range -> zero (merkle.nim:34)
    }
  }
  reinterpret_cast<uint4*>(out + 32 * ((size_t)s * max_depth + lvl))[half] = v;
}

// the raw cell of each sample whose block is in the resident tile (tile = unique blocks [first, first + ...)): order[0..n) are
// those samples, out + s * cell_size receives sample s's cell.  One thread per 4-byte word, grid-stride.
__global__ void k_gather_cells(const uint8_t* __restrict__ tile, uint64_t first, const uint32_t* __restrict__ order, size_t n,
                               const uint32_t* __restrict__ pos, const uint64_t* __restrict__ cells, uint32_t cpb_log2, uint32_t cell_size,
                               uint64_t block_size, uint8_t* __restrict__ out) {
  const uint32_t words = cell_size / 4;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n * words; t += (size_t)gridDim.x * blockDim.x) {
    const uint32_t s = order[t / words], w = (uint32_t)(t % words);
    const uint8_t* src = tile + (pos[s] - first) * block_size + (cells[s] & ((1ull << cpb_log2) - 1)) * cell_size;
    reinterpret_cast<uint32_t*>(out + (size_t)cell_size * s)[w] = reinterpret_cast<const uint32_t*>(src)[w];
  }
}

// Roofline probe: integer multiply streams, ILP 8 per thread, SASS verified (see tools/probes/probe_pipes.cu).
//   kind 0: IMAD.WIDE.U32 Rd, Ra, Rb, RZ (no carry)   kind 1: IMAD.WIDE.U32.X carry chains of 4 (exactly the
//   form of the Montgomery rows)   kind 2: 32-bit IMAD
// On B200 kinds 0 and 1 run at about half the rate of kind 2: a 32x32->64 product costs two FMA-heavy slots.
#define CDX_PROBE_OPS_PER_ITER 32
__global__ void k_probe_imad(int kind, uint32_t iters, uint32_t seed, uint32_t* __restrict__ sink) {
  uint32_t a = seed + threadIdx.x, b = seed * 3u + blockIdx.x;
  uint32_t r0 = a, r1 = b, r2 = a ^ b, r3 = a + b, r4 = a * 3, r5 = b * 5, r6 = a * 7, r7 = b * 9;
  uint32_t s0 = 1, s1 = 2, s2 = 3, s3 = 4, s4 = 5, s5 = 6, s6 = 7, s7 = 8;
  if (kind == 0) {
    // (lo,hi) = r_i * b ; r_i = lo ^ hi : each product feeds the next multiplicand, so ptxas can neither hoist the
    // multiply nor re-associate an accumulation into IADD3 chains (it does both to `acc += a*b`)
    for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        uint64_t p0 = (uint64_t)r0 * b, p1 = (uint64_t)r1 * b, p2 = (uint64_t)r2 * b, p3 = (uint64_t)r3 * b;
        uint64_t p4 = (uint64_t)r4 * b, p5 = (uint64_t)r5 * b, p6 = (uint64_t)r6 * b, p7 = (uint64_t)r7 * b;
        r0 = (uint32_t)p0 ^ (uint32_t)(p0 >> 32); r1 = (uint32_t)p1 ^ (uint32_t)(p1 >> 32);
        r2 = (uint32_t)p2 ^ (uint32_t)(p2 >> 32); r3 = (uint32_t)p3 ^ (uint32_t)(p3 >> 32);
        r4 = (uint32_t)p4 ^ (uint32_t)(p4 >> 32); r5 = (uint32_t)p5 ^ (uint32_t)(p5 >> 32);
        r6 = (uint32_t)p6 ^ (uint32_t)(p6 >> 32); r7 = (uint32_t)p7 ^ (uint32_t)(p7 >> 32);
      }
    }
  } else if (kind == 1) {
    for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
      for (int u = 0; u < 4; ++u)
        asm volatile(
            "mad.lo.cc.u32 %0,%16,%17,%0; madc.hi.cc.u32 %8,%16,%17,%8; madc.lo.cc.u32 %1,%16,%17,%1; madc.hi.cc.u32 %9,%16,%17,%9;\n\t"
            "madc.lo.cc.u32 %2,%16,%17,%2; madc.hi.cc.u32 %10,%16,%17,%10; madc.lo.cc.u32 %3,%16,%17,%3; madc.hi.u32 %11,%16,%17,%11;\n\t"
            "mad.lo.cc.u32 %4,%16,%17,%4; madc.hi.cc.u32 %12,%16,%17,%12; madc.lo.cc.u32 %5,%16,%17,%5; madc.hi.cc.u32 %13,%16,%17,%13;\n\t"
            "madc.lo.cc.u32 %6,%16,%17,%6; madc.hi.cc.u32 %14,%16,%17,%14; madc.lo.cc.u32 %7,%16,%17,%7; madc.hi.u32 %15,%16,%17,%15;"
            : "+r"(r0), "+r"(r1), "+r"(r2), "+r"(r3), "+r"(r4), "+r"(r5), "+r"(r6), "+r"(r7), "+r"(s0), "+r"(s1), "+r"(s2),
              "+r"(s3), "+r"(s4), "+r"(s5), "+r"(s6), "+r"(s7)
            : "r"(a), "r"(b));
    }
  } else {
    for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
      for (int u = 0; u < 4; ++u)
        asm volatile(
            "mad.lo.u32 %0,%0,%8,%9; mad.lo.u32 %1,%1,%8,%9; mad.lo.u32 %2,%2,%8,%9; mad.lo.u32 %3,%3,%8,%9;\n\t"
            "mad.lo.u32 %4,%4,%8,%9; mad.lo.u32 %5,%5,%8,%9; mad.lo.u32 %6,%6,%8,%9; mad.lo.u32 %7,%7,%8,%9;"
            : "+r"(r0), "+r"(r1), "+r"(r2), "+r"(r3), "+r"(r4), "+r"(r5), "+r"(r6), "+r"(r7)
            : "r"(a), "r"(b));
    }
  }
  uint32_t acc = r0 ^ r1 ^ r2 ^ r3 ^ r4 ^ r5 ^ r6 ^ r7 ^ s0 ^ s1 ^ s2 ^ s3 ^ s4 ^ s5 ^ s6 ^ s7;
  if (acc == 0x12345678u) sink[0] = acc;   // never true in practice; keeps the loop alive
}

}  // namespace cdx
