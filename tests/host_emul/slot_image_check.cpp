// The import-time header checks of slot images (csrc/slot_image.h) behind a flat C entry point, so the tests can drive
// them with g++ alone.  out receives: compact, cell_size, block_size, n_blocks, n_bytes, n_cells, cpb, block_depth,
// slot_depth, forest_nodes, top_nodes, level0_nodes, forest_width[33], slot_width[40].
#include <initializer_list>

#include "../../codex-storage-proofs-circuits_b200/csrc/slot_image.h"

extern "C" int image_layout(const uint8_t* header, uint64_t image_bytes, uint64_t* out, char* msg, size_t cap) {
  SlotImageLayout L;
  const int rc = slot_image_layout(header, image_bytes, &L, msg, cap);
  if (rc) return rc;
  uint64_t* o = out;
  for (uint64_t v : {(uint64_t)L.compact, L.cell_size, L.block_size, L.n_blocks, L.n_bytes, L.n_cells, L.cpb, (uint64_t)L.block_depth,
                     (uint64_t)L.slot_depth, L.forest_nodes, L.top_nodes, L.level0_nodes})
    *o++ = v;
  for (uint64_t v : L.forest_width) *o++ = v;
  for (uint64_t v : L.slot_width) *o++ = v;
  return rc;
}
