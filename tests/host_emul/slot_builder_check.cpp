// The bookkeeping and argument checks of the slot builder (csrc/slot_builder.h) behind flat C entry points, so the tests can
// drive them with g++ alone.  book_finish marks the book finished when finish may build the slot, as a successful
// cdx_slot_builder_finish does.
#include "../../codex-storage-proofs-circuits_b200/csrc/slot_builder.h"

extern "C" {

int builder_shape(uint64_t n_blocks, uint64_t cell_size, uint64_t block_size, char* msg, size_t cap) {
  return slot_builder_shape(n_blocks, cell_size, block_size, msg, cap);
}

void* book_new(uint64_t n_blocks) {
  SlotBuilderBook* B = new SlotBuilderBook;
  slot_builder_init(B, n_blocks);
  return B;
}

void book_free(void* B) { delete static_cast<SlotBuilderBook*>(B); }

int book_add(void* B, uint64_t first_block, uint64_t n_bytes, uint64_t block_size, uint64_t* n_out, char* msg, size_t cap) {
  return slot_builder_add(static_cast<SlotBuilderBook*>(B), first_block, n_bytes, block_size, n_out, msg, cap);
}

uint64_t book_missing(void* B, uint64_t* smallest) { return slot_builder_missing(static_cast<SlotBuilderBook*>(B), smallest); }

int book_finish(void* B, char* msg, size_t cap) {
  SlotBuilderBook* book = static_cast<SlotBuilderBook*>(B);
  const int rc = slot_builder_finish_status(book, msg, cap);
  if (rc == CDX_OK) book->finished = true;
  return rc;
}

}  // extern "C"
