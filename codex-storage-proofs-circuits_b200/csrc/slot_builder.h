// slot_builder.h -- the argument checks and the bookkeeping of a slot builder (cdx_slot_builder_*): which blocks have been
// added, whether an add may be taken, what is still missing at finish.  Host code only, no CUDA: the same header is
// compiled on its own by the tests.
//
// Every range is checked without overflow: first_block + n may wrap 64 bits for a caller-supplied first_block, and
// n_blocks * block_size may wrap for a caller-supplied shape.  A refused add changes nothing; an accepted one marks its
// blocks before any byte of it is copied.
#pragma once
#include <cstdint>
#include <vector>

#include "slot_image.h"

struct SlotBuilderBook {
  uint64_t n_blocks = 0;
  uint64_t n_added = 0;
  bool finished = false;          // set after a successful finish: every later add is refused
  std::vector<uint64_t> bits;     // bit b of word b / 64: block b has been added
};

// the shape of a builder's slot: the rules of a commit of n_blocks * block_size bytes, and a product that does not wrap
static inline int slot_builder_shape(uint64_t n_blocks, uint64_t cell_size, uint64_t block_size, char* msg, size_t cap) {
  uint64_t n_bytes = 0;
  if (__builtin_mul_overflow(n_blocks, block_size, &n_bytes))
    return slot_image_say(msg, cap, CDX_ERR_SIZE, "slot builder: %llu blocks of %llu bytes overflow 64 bits", (unsigned long long)n_blocks,
                          (unsigned long long)block_size);
  return slot_shape_status(n_bytes, cell_size, block_size, msg, cap);
}

static inline void slot_builder_init(SlotBuilderBook* B, uint64_t n_blocks) {
  B->n_blocks = n_blocks;
  B->n_added = 0;
  B->finished = false;
  B->bits.assign((size_t)((n_blocks + 63) / 64), 0);
}

static inline bool slot_builder_has(const SlotBuilderBook* B, uint64_t b) { return (B->bits[(size_t)(b >> 6)] >> (b & 63)) & 1u; }

// the smallest added block of [first, first + n) (a range inside the slot), or false if there is none
static inline bool slot_builder_first_added(const SlotBuilderBook* B, uint64_t first, uint64_t n, uint64_t* block) {
  uint64_t b = first;
  const uint64_t end = first + n;
  while (b < end) {
    const uint64_t w = B->bits[(size_t)(b >> 6)] >> (b & 63);          // the rest of b's word, from b on
    if (w) {
      const uint64_t hit = b + (uint64_t)__builtin_ctzll(w);
      if (hit < end) {
        *block = hit;
        return true;
      }
      return false;
    }
    b = (b | 63) + 1;
  }
  return false;
}

// Checks an add of n_bytes at first_block and, if it is taken, marks its blocks.  Status order: after finish (STATE), size
// (SIZE), range (RANGE), a block already added (STATE, naming the smallest one).  *n_out = the number of blocks.
static inline int slot_builder_add(SlotBuilderBook* B, uint64_t first_block, uint64_t n_bytes, uint64_t block_size, uint64_t* n_out, char* msg,
                                   size_t cap) {
  if (B->finished) return slot_image_say(msg, cap, CDX_ERR_STATE, "slot builder: the slot is finished, no block can be added");
  if (n_bytes == 0 || n_bytes % block_size)
    return slot_image_say(msg, cap, CDX_ERR_SIZE, "slot builder: an add of %llu bytes is not a non-zero multiple of the block size %llu",
                          (unsigned long long)n_bytes, (unsigned long long)block_size);
  const uint64_t n = n_bytes / block_size;
  if (first_block >= B->n_blocks || n > B->n_blocks - first_block)
    return slot_image_say(msg, cap, CDX_ERR_RANGE, "slot builder: blocks [%llu,+%llu) are outside the slot of %llu blocks", (unsigned long long)first_block,
                          (unsigned long long)n, (unsigned long long)B->n_blocks);
  uint64_t dup = 0;
  if (slot_builder_first_added(B, first_block, n, &dup))
    return slot_image_say(msg, cap, CDX_ERR_STATE, "slot builder: block %llu has already been added", (unsigned long long)dup);
  for (uint64_t b = first_block; b < first_block + n;) {
    const uint64_t in = b & 63, take = n - (b - first_block) < 64 - in ? n - (b - first_block) : 64 - in;
    B->bits[(size_t)(b >> 6)] |= (take == 64 ? ~0ull : ((1ull << take) - 1)) << in;
    b += take;
  }
  B->n_added += n;
  *n_out = n;
  return CDX_OK;
}

// the number of blocks not added yet and the smallest of them (n_blocks when none is missing)
static inline uint64_t slot_builder_missing(const SlotBuilderBook* B, uint64_t* smallest) {
  *smallest = B->n_blocks;
  for (size_t w = 0; w < B->bits.size(); ++w) {
    uint64_t free_bits = ~B->bits[w];
    if (w + 1 == B->bits.size() && B->n_blocks % 64) free_bits &= (1ull << (B->n_blocks % 64)) - 1;
    if (free_bits) {
      *smallest = 64 * (uint64_t)w + (uint64_t)__builtin_ctzll(free_bits);
      break;
    }
  }
  return B->n_blocks - B->n_added;
}

// finish may build the slot: CDX_OK, or CDX_ERR_STATE after a successful finish or with blocks missing
static inline int slot_builder_finish_status(const SlotBuilderBook* B, char* msg, size_t cap) {
  if (B->finished) return slot_image_say(msg, cap, CDX_ERR_STATE, "slot builder: the slot is finished already");
  uint64_t smallest = 0;
  const uint64_t missing = slot_builder_missing(B, &smallest);
  if (missing)
    return slot_image_say(msg, cap, CDX_ERR_STATE, "slot builder: %llu of %llu blocks are missing, the smallest is block %llu", (unsigned long long)missing,
                          (unsigned long long)B->n_blocks, (unsigned long long)smallest);
  return CDX_OK;
}
