// slot_image.h -- the header of a persisted slot image (cdx_slot_export / cdx_slot_import) and every check import makes on
// it before anything is allocated.  Host code only, no CUDA: the same header is compiled on its own by the tests.
//
// An image comes from disk, so every field is untrusted.  slot_image_layout maps (header, image length) either to the
// layout of the slot it describes -- the widths of every retained level -- or to a status and a message.  Every size is
// computed with an overflow check: a header whose node counts wrap 64 bits could otherwise describe a 2^59-block slot in
// a 2 KB file and make later calls read far outside the allocations sized from it.
#pragma once
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../include/codex_commit.h"

// A full image ("CDXSLOT1") holds the block forest and slot levels 1..depth; a compact image ("CDXSLOTC", forest_nodes = 0)
// holds slot levels 0..depth, i.e. the block hashes and everything above them.
struct SlotImageHeader {
  char magic[8];              // "CDXSLOT1" or "CDXSLOTC"
  uint64_t cell_size, block_size, n_blocks, forest_nodes, top_nodes;
  uint32_t block_depth, slot_depth;
};
static_assert(sizeof(SlotImageHeader) == 56, "the image header is 56 bytes on every platform");

// The deepest trees a proof call can answer for (PathPlan in kernels.cuh: 32 block-forest levels, 40 slot-tree levels).
#define CDX_MAX_BLOCK_DEPTH 32u
#define CDX_MAX_SLOT_DEPTH 39u

struct SlotImageLayout {
  bool compact;
  uint64_t cell_size, block_size, n_blocks, n_bytes, n_cells, cpb;
  uint32_t block_depth, slot_depth;
  uint64_t forest_width[CDX_MAX_BLOCK_DEPTH + 1];   // block-forest level l over all blocks, l = 0..block_depth (full images)
  uint64_t slot_width[CDX_MAX_SLOT_DEPTH + 1];      // slot-tree level l, l = 0..slot_depth
  uint64_t forest_nodes;                            // forest levels 0..block_depth as stored (0 in a compact image)
  uint64_t top_nodes;                               // slot levels 1..slot_depth
  uint64_t level0_nodes;                            // what precedes slot level 1 in the payload
};

static inline int slot_image_say(char* msg, size_t cap, int status, const char* fmt, ...) {
  if (msg && cap) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(msg, cap, fmt, ap);
    va_end(ap);
  }
  return status;
}

// the cell and block sizes a slot may have and its size in bytes: CDX_OK, or CDX_ERR_SIZE with a message
static inline int slot_shape_status(uint64_t n_bytes, uint64_t cell_size, uint64_t block_size, char* msg, size_t cap) {
  if (cell_size == 0 || cell_size % 4 || cell_size > (1u << 30))
    return slot_image_say(msg, cap, CDX_ERR_SIZE, "cell size %llu must be a non-zero multiple of 4", (unsigned long long)cell_size);
  if (block_size == 0 || block_size % cell_size) return slot_image_say(msg, cap, CDX_ERR_SIZE, "block size is not divisible by cell size");
  const uint64_t cpb = block_size / cell_size;
  if (cpb & (cpb - 1)) return slot_image_say(msg, cap, CDX_ERR_SIZE, "cells per block (%llu) must be a power of two", (unsigned long long)cpb);
  if (n_bytes == 0 || n_bytes % block_size)
    return slot_image_say(msg, cap, CDX_ERR_SIZE, "slot size %llu is not a non-zero multiple of the block size", (unsigned long long)n_bytes);
  return CDX_OK;
}

// Status order: too short for a header (SIZE), magic (ARG), shape and a slot size that overflows (SIZE), depths that
// disagree with the geometry (ARG), depths beyond CDX_MAX_*_DEPTH (RANGE), forest_nodes (ARG, SIZE on overflow), top_nodes
// and the image length (SIZE).
static inline int slot_image_layout(const void* image, uint64_t image_bytes, SlotImageLayout* L, char* msg, size_t cap) {
  SlotImageHeader h;
  if (image_bytes < sizeof h) return slot_image_say(msg, cap, CDX_ERR_SIZE, "image too small");
  memcpy(&h, image, sizeof h);
  memset(L, 0, sizeof *L);
  L->compact = memcmp(h.magic, "CDXSLOTC", 8) == 0;
  if (!L->compact && memcmp(h.magic, "CDXSLOT1", 8) != 0) return slot_image_say(msg, cap, CDX_ERR_ARG, "not a slot image");
  if (__builtin_mul_overflow(h.n_blocks, h.block_size, &L->n_bytes))
    return slot_image_say(msg, cap, CDX_ERR_SIZE, "slot image: %llu blocks of %llu bytes overflow 64 bits", (unsigned long long)h.n_blocks,
                          (unsigned long long)h.block_size);
  const int rc = slot_shape_status(L->n_bytes, h.cell_size, h.block_size, msg, cap);
  if (rc) return rc;
  L->cell_size = h.cell_size;
  L->block_size = h.block_size;
  L->n_blocks = h.n_blocks;
  L->cpb = h.block_size / h.cell_size;
  L->n_cells = L->n_bytes / h.cell_size;                 // = n_blocks * cpb, exact
  uint32_t cpb_log2 = 0;
  while ((1ull << cpb_log2) < L->cpb) ++cpb_log2;
  const uint32_t block_depth = L->cpb == 1 ? 1 : cpb_log2;
  // slot-tree widths n, ceil(n/2), ..., 1; a single block still gets one key-3 compression (merkle/bn254.nim:29-60)
  uint32_t slot_depth = 0;
  for (uint64_t w = h.n_blocks; slot_depth == 0 || w > 1; w = w / 2 + (w & 1)) {
    if (slot_depth <= CDX_MAX_SLOT_DEPTH) L->slot_width[slot_depth] = w;
    ++slot_depth;
  }
  if (slot_depth <= CDX_MAX_SLOT_DEPTH) L->slot_width[slot_depth] = 1;
  if (h.block_depth != block_depth || h.slot_depth != slot_depth)
    return slot_image_say(msg, cap, CDX_ERR_ARG, "slot image header is inconsistent with its geometry: depths %u and %u, the geometry gives %u and %u",
                          h.block_depth, h.slot_depth, block_depth, slot_depth);
  if (block_depth > CDX_MAX_BLOCK_DEPTH || slot_depth > CDX_MAX_SLOT_DEPTH)
    return slot_image_say(msg, cap, CDX_ERR_RANGE, "slot image: trees of depth %u and %u are too deep for the path plan (at most %u and %u)",
                          block_depth, slot_depth, CDX_MAX_BLOCK_DEPTH, CDX_MAX_SLOT_DEPTH);
  L->block_depth = block_depth;
  L->slot_depth = slot_depth;
  uint64_t forest = 0;
  for (uint32_t l = 0; l <= block_depth; ++l) {
    L->forest_width[l] = L->cpb == 1 ? L->n_cells : (L->n_cells >> l);
    if (__builtin_add_overflow(forest, L->forest_width[l], &forest))
      return slot_image_say(msg, cap, CDX_ERR_SIZE, "slot image: the block forest's node count overflows 64 bits");
  }
  L->forest_nodes = L->compact ? 0 : forest;
  if (h.forest_nodes != L->forest_nodes)
    return slot_image_say(msg, cap, CDX_ERR_ARG, "slot image header is inconsistent with its geometry: forest_nodes %llu, the geometry gives %llu",
                          (unsigned long long)h.forest_nodes, (unsigned long long)L->forest_nodes);
  for (uint32_t l = 1; l <= slot_depth; ++l) L->top_nodes += L->slot_width[l];   // < 2 n_blocks: no overflow
  L->level0_nodes = L->compact ? L->slot_width[0] : L->forest_nodes;
  uint64_t nodes, bytes;
  if (h.top_nodes != L->top_nodes || __builtin_add_overflow(L->level0_nodes, L->top_nodes, &nodes) || __builtin_mul_overflow(nodes, (uint64_t)32, &bytes) ||
      __builtin_add_overflow(bytes, (uint64_t)sizeof h, &bytes) || bytes != image_bytes)
    return slot_image_say(msg, cap, CDX_ERR_SIZE, "slot image has the wrong length");
  return CDX_OK;
}
