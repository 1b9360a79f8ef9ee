/* codex_commit.h -- C ABI of libcodexcommit.so, the B200 (sm_100a) slot-commitment backend.
 *
 * The reference (codex-storage-proofs-circuits, reference/nim/proof_input) has no FFI seam of its own: its
 * arithmetic comes from the Nim packages `poseidon2` and `constantine`, called from a handful of places.  The
 * entry points below are exactly what a Nim `importc` binding would need to replace those call sites and the
 * loops around them; each one cites the reference interface it stands in for (file:line under /root/reference,
 * `nim/` = reference/nim/proof_input/src/).  INTEGRATION.md shows the Nim-side stub.
 *
 * Conventions
 *   - A field element (Nim `F`, `Hash`, `Root`, `Entropy`: nim/types/bn254.nim:20-23) crosses the ABI as 32 bytes,
 *     little-endian, canonical (value < r).  Inputs >= r are taken mod r.  Outputs are always canonical.
 *   - The caller owns every buffer.  `_host` entry points take host pointers and perform the transfers
 *     themselves; `_dev` entry points take CUDA device pointers and a cudaStream_t (as void*) and are
 *     asynchronous with respect to the host.
 *   - Every function returns 0 (CDX_OK) or a negative cdx_status; nothing aborts (the reference asserts:
 *     nim/blocks/bn254.nim:26,34, nim/sample/bn254.nim:20).  cdx_last_error(ctx) gives the message.
 *   - One cdx_ctx per (host thread, GPU).  Handles are not shared between threads.
 *   - There is NO CPU implementation behind this ABI: without a CUDA device cdx_ctx_create fails with
 *     CDX_ERR_CUDA and nothing else can be called.
 */
#ifndef CODEX_COMMIT_H
#define CODEX_COMMIT_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CDX_ABI_VERSION 2
#define CDX_FELT_BYTES 32

typedef enum cdx_status {
  CDX_OK = 0,
  CDX_ERR_ARG = -1,      /* null pointer, zero count, bad rate/key */
  CDX_ERR_SIZE = -2,     /* sizes not divisible as the reference asserts (nim/types.nim:120-123, nim/blocks/bn254.nim:26,34) */
  CDX_ERR_NOT_POW2 = -3, /* numberOfCells must be a power of two (nim/sample/bn254.nim:19-20) */
  CDX_ERR_RANGE = -4,    /* index out of range (nim/merkle.nim:27) or depth too small (nim/types.nim:29) */
  CDX_ERR_CUDA = -5,     /* CUDA runtime error, or no device */
  CDX_ERR_ALLOC = -6,
  CDX_ERR_STATE = -7,    /* handle not in the state the call needs (e.g. sharded slot without its top tree) */
  CDX_ERR_MISMATCH = -8  /* slot bytes do not hash to the retained commitment (cdx_slot_prove_from_source), or a node
                            of a slot image does not hash from its children or is not canonical (cdx_slot_import) */
} cdx_status;

typedef struct cdx_ctx cdx_ctx;   /* per-GPU context: device, streams, staging buffers */
typedef struct cdx_slot cdx_slot; /* a committed slot: every Merkle layer resident in HBM */

/* ---- context ------------------------------------------------------------------------------------------ */
int cdx_abi_version(void);
/* number of CUDA devices this process can see (0 without a driver or a device); creates no context */
int cdx_device_count(void);
int cdx_ctx_create(int device, cdx_ctx** out);
void cdx_ctx_destroy(cdx_ctx* ctx);
const char* cdx_last_error(const cdx_ctx* ctx);
const char* cdx_status_string(int status);
/* number of kernels this context has launched since creation (bench.py's gpu_launches) */
uint64_t cdx_launch_count(const cdx_ctx* ctx);
/* the CUDA stream (cudaStream_t) host-pointer entry points run on; lets callers time them with events */
void* cdx_ctx_stream(const cdx_ctx* ctx);

/* ---- hash layer (what nim-poseidon2 provides to the reference) ------------------------------------------ */

/* n independent Poseidon2 permutations, 3 elements in / 3 out each.
 * Replaces: permutation, reference/haskell/src/Poseidon2/Permutation.hs:40-45 (Nim: poseidon2 `perm`). */
int cdx_permutation_batch_host(cdx_ctx* ctx, const uint8_t* in, uint8_t* out, size_t n);
int cdx_permutation_batch_dev(cdx_ctx* ctx, const void* d_in, void* d_out, size_t n, void* stream);

/* n_items sponges, each over `len` field elements (item i at elems + i*len*32), rate 1 or 2.
 * Replaces: Sponge.digest(openArray[F], rate) -- nim/sample/bn254.nim:23, testvectors.nim:26,34;
 * reference/haskell/src/Poseidon2/Sponge.hs:13-43. */
int cdx_sponge_felts_batch_host(cdx_ctx* ctx, const uint8_t* elems, size_t n_items, size_t len, int rate, uint8_t* out);

/* n_items byte strings of equal length `len` (item i at data + i*len), each hashed with the rate-2 sponge after
 * 31-byte 10* chunking.  Replaces: Sponge.digest(openArray[byte], rate=2) -- nim/blocks/bn254.nim:27 (hashCell),
 * testvectors.nim:45; reference/haskell/src/Slot.hs:222-270. */
int cdx_hash_bytes_batch_host(cdx_ctx* ctx, const uint8_t* data, size_t n_items, size_t len, uint8_t* out);

/* Cell hashes only, device to device: n_cells cells of cell_size bytes (a multiple of 4) at d_data -> n_cells field
 * elements at d_out.  This is the dominant kernel of the path (34 permutations per 2048-byte cell); bench.py times
 * it alone for the roofline.  Replaces: the hashCell loop of networkBlockTree -- nim/blocks/bn254.nim:23-29,63. */
int cdx_hash_cells_dev(cdx_ctx* ctx, const void* d_data, size_t n_cells, size_t cell_size, void* d_out, void* stream);

/* out[i] = perm(x[i], y[i], keys[i])[0], keys in 0..3.
 * Replaces: compress(x, y, key=) via compressWithkey -- nim/merkle/bn254.nim:18,50,53;
 * reference/haskell/src/Poseidon2/Merkle.hs:202-203. */
int cdx_compress_batch_host(cdx_ctx* ctx, const uint8_t* x, const uint8_t* y, const uint32_t* keys, size_t n, uint8_t* out);

/* ---- Merkle trees --------------------------------------------------------------------------------------- */

/* Total node count over all layers of a tree with n leaves (layers n, ceil(n/2), ..., 1).  With
 * bottom_layer != 0 a single leaf still gets one key-3 compression (2 layers); otherwise a single node is its
 * own root.  Mirrors merkleTreeWorker, nim/merkle/bn254.nim:29-60. */
size_t cdx_merkle_total_nodes(size_t n, int bottom_layer);
int cdx_merkle_num_layers(size_t n, int bottom_layer);

/* All layers bottom-first, concatenated, into layers_out (cdx_merkle_total_nodes(n) * 32 bytes).
 * Replaces: merkleTreeBN254 / merkleTree -- nim/merkle/bn254.nim:62-63, nim/blocks/bn254.nim:17-19;
 * reference/haskell/src/Poseidon2/Merkle.hs:69-83.  Key rule: bit0 = first level only, bit1 = odd node
 * (single child paired with 0), single leaf = one key-3 compression. */
int cdx_merkle_layers_host(cdx_ctx* ctx, const uint8_t* leaves, size_t n, int bottom_layer, uint8_t* layers_out);

/* Root only.  Replaces: Merkle.digest / merkleDigestBN254 -- nim/merkle/bn254.nim:20, testvectors.nim:56. */
int cdx_merkle_root_host(cdx_ctx* ctx, const uint8_t* leaves, size_t n, uint8_t root_out[32]);

/* Merkle.digest over a byte string: the bytes are chunked into field elements exactly like a cell (31-byte little-endian
 * chunks of data ++ 0x01 ++ 0x00.., floor(len/31)+1 elements) and those elements are the leaves of the tree.
 * Replaces: Merkle.digest(openArray[byte]) -- reference/nim/testvectors/src/testvectors.nim:60-66 (n = 0..80). */
int cdx_merkle_root_bytes_host(cdx_ctx* ctx, const uint8_t* data, size_t len, uint8_t root_out[32]);


/* ---- slot commitment ------------------------------------------------------------------------------------ */

/* Commit a whole slot: hash every cell (34 permutations per 2048-byte cell), build every block tree
 * (cells_per_block leaves each), then the slot tree over the block hashes.  All layers stay in HBM inside the
 * returned handle so that paths can be extracted later without rehashing.
 * Replaces: buildSlotTreeFull -- nim/gen_input/bn254.nim:21-30 (hashCell, networkBlockTree, merkleTree);
 * reference/haskell/src/Slot.hs:151-179.
 * Requirements (else CDX_ERR_SIZE): cell_size a multiple of 4, block_size a multiple of cell_size with a
 * power-of-two quotient, n_bytes a non-zero multiple of block_size. */
int cdx_slot_commit_host(cdx_ctx* ctx, const uint8_t* data, size_t n_bytes, size_t cell_size, size_t block_size, cdx_slot** out);
int cdx_slot_commit_dev(cdx_ctx* ctx, const void* d_data, size_t n_bytes, size_t cell_size, size_t block_size, void* stream, cdx_slot** out);

/* Commit a slot straight from a file: bytes [offset, offset + n_bytes) of `path` stream through pinned host buffers
 * (parallel pread) -> H2D -> cell sponge, all three overlapped; only the hashes stay resident.  Bytes past the end of
 * the file read as zeros, like the reference's ignored short reads.
 * Replaces: slotLoadCellData(SlotFile) + buildSlotTreeFull -- nim/slot.nim:57-68 (one open/seek/read per 2 KiB cell),
 * nim/dataset.nim:34-41, nim/gen_input/bn254.nim:21-30.  (SURVEY.md 8f item 1.) */
int cdx_slot_commit_file(cdx_ctx* ctx, const char* path, uint64_t offset, size_t n_bytes, size_t cell_size, size_t block_size, cdx_slot** out);

/* Same over the reference's fake data source, generated on the device (never crosses PCIe).
 * Replaces: slotLoadBlockData + genFakeCell -- nim/slot.nim:23-32,70-73, seed as in nim/dataset.nim:32. */
int cdx_slot_commit_fake(cdx_ctx* ctx, uint64_t seed, size_t n_cells, size_t cell_size, size_t block_size, cdx_slot** out);

/* Sharded commitment (one process per GPU).  This rank holds blocks [first_block, first_block + n_local_blocks)
 * of a slot of n_total_blocks; first_block must be a multiple of 2^top_level, and so must n_local_blocks unless
 * the range ends at n_total_blocks.  Levels 0..top_level of the slot tree are built for the local range; the
 * level-top_level nodes are the sub-tree roots to exchange (cdx_slot_exchange_top does it over NCCL; these calls are the
 * pieces it is made of, for hosts that bring their own transport).  cdx_slot_set_top then installs the
 * gathered level and builds the replicated upper levels.  (The reference is single-process; the tree
 * conventions are nim/merkle/bn254.nim:29-60 with the odd-node rule applied to the GLOBAL layer width.) */
int cdx_slot_commit_range_dev(cdx_ctx* ctx, const void* d_data, size_t n_local_bytes, size_t cell_size, size_t block_size,
                              uint64_t first_block, uint64_t n_total_blocks, int top_level, void* stream, cdx_slot** out);
int cdx_slot_commit_range_host(cdx_ctx* ctx, const uint8_t* data, size_t n_local_bytes, size_t cell_size, size_t block_size,
                               uint64_t first_block, uint64_t n_total_blocks, int top_level, cdx_slot** out);
int cdx_slot_subtree_root_count(const cdx_slot* slot, uint64_t* first_node, uint64_t* n_nodes);
/* copy this rank's level-top_level nodes into a caller buffer (a host-provided transport's send buffer) */
int cdx_slot_subtree_roots_copy_dev(const cdx_slot* slot, void* d_dst, void* stream);
/* device pointer to this rank's level-top_level nodes (n_nodes * 32 bytes), for NCCL */
const void* cdx_slot_subtree_roots_dev(const cdx_slot* slot);
int cdx_slot_set_top_dev(cdx_slot* slot, const void* d_level_nodes, uint64_t n_level_nodes, void* stream);

/* Persist / restore a commitment (SURVEY.md 8f item 2: a proof server answers repeated challenges from a retained
 * commitment instead of re-hashing the slot).  The image is a small header followed by every retained layer (canonical
 * 32-byte elements), about 3.1 % of the slot size; it is self-describing.  Only whole
 * (non-sharded, top tree present) slots can be exported.  The reference keeps nothing: it rebuilds the slot tree for
 * every sample (nim/gen_input/bn254.nim:57).
 * A compact slot (cdx_slot_compact) exports a compact image: magic "CDXSLOTC", forest_nodes = 0, slot-tree levels
 * 0..slot_tree_depth (32 bytes x the sum of their widths, about 0.1 % of the slot at the default geometry); importing it
 * gives a compact slot.
 * Import checks the image before it returns a handle.  First the header, before anything is allocated: the magic
 * (CDX_ERR_ARG); the cell and block sizes as a commit checks them and sizes that would overflow 64 bits (CDX_ERR_SIZE);
 * depths and forest_nodes that disagree with the geometry (CDX_ERR_ARG); trees deeper than a proof call can answer for,
 * block_tree_depth > 32 or slot_tree_depth > 39 (CDX_ERR_RANGE); top_nodes and the image length (CDX_ERR_SIZE).
 * Then the payload, on the device:
 * every stored node above the bottom level must be the compression of its stored children, and every stored element
 * must be canonical (< r); otherwise CDX_ERR_MISMATCH, and the message names the smallest bad node (tree, level, node).
 * So an imported slot is internally consistent; that its root is the root the caller expects is for the caller to
 * compare (cdx_slot_root). */
size_t cdx_slot_export_size(const cdx_slot* slot);
int cdx_slot_export(const cdx_slot* slot, uint8_t* image, size_t image_bytes);
int cdx_slot_import(cdx_ctx* ctx, const uint8_t* image, size_t image_bytes, cdx_slot** out);

void cdx_slot_free(cdx_slot* slot);

/* treeRoot of the slot tree -- nim/merkle.nim:14-17. */
int cdx_slot_root(const cdx_slot* slot, uint8_t root_out[32]);
/* shape of the retained trees */
int cdx_slot_shape(const cdx_slot* slot, uint64_t* n_cells, uint64_t* n_blocks, uint32_t* block_tree_depth, uint32_t* slot_tree_depth);
/* Copy `count` nodes starting at `first` out of a retained layer.  tree 0 = the forest of block trees
 * (level 0 = cell hashes ... level block_tree_depth = block hashes), tree 1 = the slot tree (level 0 = block
 * hashes ... level slot_tree_depth = root).  For a sharded slot, indices are global; only locally held nodes
 * (or replicated upper levels) can be read.  Mirrors MerkleTree.layers, nim/types.nim:20-22. */
int cdx_slot_read_layer(const cdx_slot* slot, int tree, uint32_t level, uint64_t first, uint64_t count, uint8_t* out);

/* Batched Merkle-path extraction for sampled cells: for each cell index, the block-tree path
 * (block_tree_depth siblings) followed by the slot-tree path (slot_tree_depth siblings), out-of-range sibling =
 * 0, zero-padded to max_depth; out is n_samples * max_depth * 32 bytes; leaf_out (may be NULL) gets the cell
 * hashes.  Replaces, per sample: merkleProof x2, mergeMerkleProofs' path concat, padMerkleProof --
 * nim/merkle.nim:21-42,86-100, nim/types.nim:27-37, nim/gen_input/bn254.nim:56-63.
 * For a sharded slot only levels held by this rank are filled, the rest are left zero (sum over ranks = path). */
int cdx_slot_cell_paths(const cdx_slot* slot, const uint64_t* cell_indices, size_t n_samples, size_t max_depth, uint8_t* out, uint8_t* leaf_out);

/* Proof-server call: answer n_challenges challenges against one retained commitment in one pass.  For challenge k
 * (entropies + 32 k) it produces what cdx_cell_indices followed by cdx_slot_cell_paths would: indices_out[k * n_samples
 * + c-1], paths_out[(k * n_samples + c-1) * max_depth * 32 ...], leaves_out (may be NULL) likewise -- the indices are
 * derived from the slot root on the device and never visit the host in between.  The slot's cell count must be a
 * power of two (nim/sample/bn254.nim:19-20).  Replaces, per challenge: cellIndices (nim/sample/bn254.nim:26-27) and
 * the per-sample proof loop of generateProofInput (nim/gen_input/bn254.nim:53-74), which rebuilds the slot tree for
 * every sample (:57). */
int cdx_slot_prove_batch(const cdx_slot* slot, const uint8_t* entropies, size_t n_challenges, size_t n_samples, size_t max_depth,
                         uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out);

/* Batched verifier walk: roots_out[i] = the root reconstructed from leaf i at index indices[i] in a tree of n_leaves
 * leaves along the first `depth` elements of its path (paths are n x path_stride elements, so padded paths can be
 * passed as they are).  Replaces: reconstructRoot / checkMerkleProof -- nim/merkle.nim:51-77 (also the check inside
 * mergeMerkleProofs, :88-89); same semantics as RootFromMerklePath, circuit/codex/merkle.circom:44-114. */
int cdx_reconstruct_roots_host(cdx_ctx* ctx, const uint8_t* leaves, const uint64_t* indices, uint64_t n_leaves, const uint8_t* paths,
                               size_t path_stride, size_t depth, size_t n, uint8_t* roots_out);

/* ---- many small slots in one pass ------------------------------------------------------------------------ */

/* n_slots slots stored back to back (slot k is slot_bytes[k] bytes, a non-zero multiple of block_size) committed with ONE
 * cell-sponge launch, one launch per block-tree level over the whole forest and one launch per slot-tree level over all
 * slot trees at once (per-slot widths, per-slot odd-node rule, singleton rule for one-block slots); the n_slots roots are
 * read back once.  A 4 MiB slot alone occupies a B200 for ~2.5 ms with 64 warps; a thousand of them batched run at the
 * large-slot rate.  Only roots are produced (commit the slot that has to be sampled on its own).
 * Replaces: the `for i in 0..<nslots: buildSlotTree(...)` loop -- nim/gen_input/bn254.nim:41-47. */
int cdx_slots_commit_batch_dev(cdx_ctx* ctx, const void* d_data, const uint64_t* slot_bytes, size_t n_slots, size_t cell_size,
                               size_t block_size, void* stream, uint8_t* roots_out);
int cdx_slots_commit_batch_host(cdx_ctx* ctx, const uint8_t* data, const uint64_t* slot_bytes, size_t n_slots, size_t cell_size,
                                size_t block_size, uint8_t* roots_out);
/* the same over the reference's fake data: slot k has seed seeds[k] and n_cells cells.
 * Replaces: slotCfgFromDataSetCfg + buildSlotTree per slot -- nim/dataset.nim:32-43, nim/gen_input/bn254.nim:41-47. */
int cdx_slots_commit_batch_fake(cdx_ctx* ctx, const uint64_t* seeds, size_t n_slots, size_t n_cells, size_t cell_size, size_t block_size,
                                uint8_t* roots_out);

/* ---- several GPUs: communicators, sharded slots ------------------------------------------------------------
 * One rank per GPU (one process per GPU, or one thread per GPU inside one process).  The only exchanges on this path are
 * (a) the level-top_level nodes of a block-range-sharded slot, (b) the 32-byte slot roots of a dataset and (c) the
 * answer to a challenge travelling from the rank(s) that hold the sampled cells -- a few KB each.  They run over NCCL
 * (NVLink/NVSwitch) inside the library, on the slot's stream, without a host round trip.  libnccl.so.2 is resolved at run
 * time (dlopen; an already loaded copy, e.g. PyTorch's, is reused); a single rank needs no NCCL at all.
 * The reference is single-process and single-threaded: these entry points have no counterpart there beyond the loops
 * they parallelise (nim/gen_input/bn254.nim:21-30,41-51). */
typedef struct cdx_comm cdx_comm;
#define CDX_COMM_ID_BYTES 128
/* rank 0 creates the id and hands it to the other ranks by any host-side means (ncclGetUniqueId) */
int cdx_comm_unique_id(uint8_t id_out[CDX_COMM_ID_BYTES]);
/* collective over all ranks: joins ctx's GPU to the communicator (ncclCommInitRank).  n_ranks == 1 never touches NCCL. */
int cdx_comm_init_rank(cdx_ctx* ctx, int n_ranks, int rank, const uint8_t id[CDX_COMM_ID_BYTES], cdx_comm** out);
void cdx_comm_destroy(cdx_comm* comm);
int cdx_comm_rank(const cdx_comm* comm);
int cdx_comm_size(const cdx_comm* comm);
/* barrier on the device: returns when every rank's stream has reached this point (a 4-byte all-reduce + stream sync) */
int cdx_comm_barrier(cdx_comm* comm);

/* Split a slot of n_total_blocks blocks over n_ranks: picks the exchange level T (the largest one that still balances
 * the ranks within 1 %) and a contiguous 2^T-aligned block range per rank.  Ranks of a slot with fewer chunks than ranks
 * get an empty range (n_blocks[r] == 0) and still take part in every collective.  (SURVEY.md 8e.) */
int cdx_plan_block_ranges(uint64_t n_total_blocks, int n_ranks, int* top_level, uint64_t* first_block, uint64_t* n_blocks);
/* The exchange level caller-chosen ranges allow: the largest T such that every range starts on a multiple of 2^T and
 * every range but the one ending the slot is a multiple of 2^T long. */
int cdx_block_ranges_top_level(uint64_t n_total_blocks, int n_ranks, const uint64_t* first_block, const uint64_t* n_blocks, int* top_level);

/* Sharded commitment in one call: this rank's block range (n_local_bytes may be 0: empty shard, data may then be NULL) is
 * committed up to level top_level, the level-top_level nodes of all ranks are combined on the device (one NCCL collective
 * on the slot's stream, no host synchronisation) and the replicated top tree is built.  Collective: every rank of `comm`
 * calls it with the same n_total_blocks and top_level.  The handle then answers cdx_slot_root on every rank and
 * cdx_slot_cell_paths_sharded / cdx_slot_prove_batch_sharded collectively. */
int cdx_slot_commit_sharded_dev(cdx_ctx* ctx, cdx_comm* comm, const void* d_data, size_t n_local_bytes, size_t cell_size, size_t block_size,
                                uint64_t first_block, uint64_t n_total_blocks, int top_level, void* stream, cdx_slot** out);
int cdx_slot_commit_sharded_host(cdx_ctx* ctx, cdx_comm* comm, const uint8_t* data, size_t n_local_bytes, size_t cell_size, size_t block_size,
                                 uint64_t first_block, uint64_t n_total_blocks, int top_level, cdx_slot** out);
/* the exchange alone, for a slot committed with cdx_slot_commit_range_* (asynchronous on the slot's stream) */
int cdx_slot_exchange_top(cdx_slot* slot, cdx_comm* comm);
/* cdx_slot_cell_paths / cdx_slot_prove_batch for a sharded slot: every rank passes the same arguments and receives the
 * complete answer (the owner of a cell fills its path, the ranks' partial results are summed byte-wise on the device). */
int cdx_slot_cell_paths_sharded(const cdx_slot* slot, cdx_comm* comm, const uint64_t* cell_indices, size_t n_samples, size_t max_depth,
                                uint8_t* out, uint8_t* leaf_out);
int cdx_slot_prove_batch_sharded(const cdx_slot* slot, cdx_comm* comm, const uint8_t* entropies, size_t n_challenges, size_t n_samples,
                                 size_t max_depth, uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out);

/* ---- dataset commitment ------------------------------------------------------------------------------------ */

typedef enum cdx_source_kind {
  CDX_SRC_FAKE = 0,      /* the reference's fake data: genFakeCell with this seed (nim/slot.nim:23-32) */
  CDX_SRC_SYNTHETIC = 1, /* counter-based benchmark bytes: byte b of the slot is byte b % 8 (little-endian) of
                            splitmix64(seed + b / 8), for any slot size and any block range or batch offset; where
                            both are multiples of 8 this is word i = splitmix64(seed + i) (cdx_fill_synthetic_dev) */
  CDX_SRC_FILE = 2,      /* a slot data file, read from offset 0 (nim/dataset.nim:34: <base><k>.dat) */
  CDX_SRC_HOST = 3       /* bytes in host memory */
} cdx_source_kind;

typedef struct cdx_slot_desc {   /* one slot of a dataset (SlotConfig, nim/types.nim:75-79) */
  uint32_t kind;                 /* cdx_source_kind */
  uint32_t reserved;
  uint64_t seed;                 /* CDX_SRC_FAKE / CDX_SRC_SYNTHETIC */
  const char* path;              /* CDX_SRC_FILE */
  const uint8_t* host;           /* CDX_SRC_HOST */
  uint64_t n_bytes;              /* slot size: a non-zero multiple of block_size */
} cdx_slot_desc;

typedef struct cdx_dataset cdx_dataset;

/* Commit every slot of a dataset and build the dataset tree over the slot roots.  With a communicator (may be NULL = one
 * GPU) the slots are dealt to the ranks by longest-processing-time bin packing, slots that would unbalance the ranks are
 * block-range-sharded over all of them, small slots are committed in batches, the 32-byte roots are combined with ONE
 * collective and every rank builds the (tiny) dataset tree.  Collective: every rank passes the same arguments.
 * keep_slot (or -1): that slot's commitment is retained for cdx_dataset_prove.
 * Replaces: the slot loop, dataset tree and slot proof of generateProofInput -- nim/gen_input/bn254.nim:41-51;
 * reference/haskell/src/Sampling.hs:66-70,84. */
int cdx_dataset_commit(cdx_ctx* ctx, cdx_comm* comm, const cdx_slot_desc* slots, size_t n_slots, size_t cell_size, size_t block_size,
                       int64_t keep_slot, cdx_dataset** out);
/* The plan cdx_dataset_commit follows, without committing anything (pure host function, no GPU needed): owner_out[k] = the
 * rank that commits slot k whole (alone or in a batch), or -1 if slot k is block-range-sharded over all ranks. */
int cdx_dataset_plan(const uint64_t* slot_bytes, size_t n_slots, size_t block_size, int n_ranks, int* owner_out);
void cdx_dataset_free(cdx_dataset* ds);
int cdx_dataset_root(const cdx_dataset* ds, uint8_t root_out[32]);
/* all slot roots, n_slots * 32 bytes */
int cdx_dataset_slot_roots(const cdx_dataset* ds, uint8_t* roots_out);
/* merkleProof(dsetTree, slot_index) zero-padded to max_log2_nslots elements -- nim/gen_input/bn254.nim:50-51, nim/types.nim:27-37 */
int cdx_dataset_slot_proof(const cdx_dataset* ds, uint64_t slot_index, size_t max_log2_nslots, uint8_t* path_out);
/* bytes this rank hashed, how many slots it committed whole / in batches / as shards (diagnostics for the bench line) */
int cdx_dataset_stats(const cdx_dataset* ds, uint64_t* bytes_local, uint32_t* n_whole, uint32_t* n_batched, uint32_t* n_sharded);
/* The kept slot's handle on this rank: the whole slot on its owner, a shard on every rank if it was sharded, NULL elsewhere. */
cdx_slot* cdx_dataset_kept_slot(const cdx_dataset* ds);
/* Answer one challenge against the kept slot: cell indices from (entropy, slot root), cell hashes and merged, padded
 * Merkle paths.  Collective when the dataset was committed with a communicator; every rank receives the answer.
 * Replaces: cellIndices + the per-sample proof loop -- nim/sample/bn254.nim:26-27, nim/gen_input/bn254.nim:53-74. */
int cdx_dataset_prove(const cdx_dataset* ds, const uint8_t entropy[32], size_t n_samples, size_t max_depth, uint64_t* indices_out,
                      uint8_t* paths_out, uint8_t* leaves_out);

/* ---- compact commitments ---------------------------------------------------------------------------------
 * A challenge samples n_samples cells, and the prover reads those cells' bytes from storage anyway: they are the
 * `cellData` of the proof input (slotLoadCellData per sample, nim/gen_input/bn254.nim:53-74, nim/slot.nim:51-68).  So a
 * proof server can keep only the slot tree (the block hashes and above: 32 bytes per block and about as much again for
 * the levels above, 0.1 % of the slot at 64 KiB blocks) instead of the whole block forest (3.1 %), and rebuild the block
 * trees of the sampled blocks from their bytes at every challenge.  Doing so also checks that the stored bytes still
 * hash to the commitment.
 *
 * cdx_slot_compact: release the block forest below the block hashes of a whole slot with its top tree (CDX_ERR_STATE for a
 * shard, a range slot or a slot without its top tree; compacting a compact slot is a no-op).  Afterwards root, shape,
 * read_layer(tree 1, any level) and read_layer(tree 0, block_tree_depth) work as before; read_layer(tree 0, lower levels),
 * cdx_slot_cell_paths, cdx_slot_prove_batch and cdx_dataset_prove on a compacted kept slot return CDX_ERR_STATE.
 * cdx_slot_device_bytes: device memory the handle holds for its tree levels (a diagnostic). */
int cdx_slot_compact(cdx_slot* slot);
size_t cdx_slot_device_bytes(const cdx_slot* slot);

/* cdx_slot_prove_batch for a compact or full whole slot, from the slot's bytes: `source` describes them as a dataset slot
 * does (CDX_SRC_FAKE, CDX_SRC_SYNTHETIC, CDX_SRC_FILE read from offset 0, CDX_SRC_HOST), source->n_bytes must be the slot
 * size (else CDX_ERR_SIZE).  The cell indices are derived from the retained root; only the unique sampled blocks are read,
 * hashed into their block trees and checked against the retained block hashes.  indices_out, paths_out and leaves_out
 * (may be NULL) are byte for byte what cdx_slot_prove_batch gives on the full slot.  cells_out (may be NULL) receives the
 * raw bytes of every sampled cell, n_challenges x n_samples x cell_size bytes in (challenge, counter) order: the
 * reference's cellData before elements() (nim/gen_input/bn254.nim:53-74, nim/slot.nim:51-68).  A block whose bytes do
 * not hash to its retained hash fails the call with CDX_ERR_MISMATCH (the message names the smallest such block; the
 * outputs are then unspecified); a file that cannot be opened or read is CDX_ERR_ARG, bytes past its end read as zeros.
 * Limits as cdx_slot_prove_batch.  Returns synchronised. */
int cdx_slot_prove_from_source(const cdx_slot* slot, const cdx_slot_desc* source, const uint8_t* entropies, size_t n_challenges,
                               size_t n_samples, size_t max_depth, uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out,
                               uint8_t* cells_out);

/* cdx_slot_prove_from_source for many slots at once.  Challenge k is entropies + 32 k against slots[k], whose bytes
 * sources[k] describes (as for cdx_slot_prove_from_source).  A handle may appear in several rows; those rows must give equal
 * descriptors (kind, seed / path / host pointer, n_bytes), and each of its sampled blocks is read and hashed once for all of them.
 * Outputs use the layout of cdx_slot_prove_from_source with n_challenges rows: indices_out[k * n_samples + c - 1], paths_out,
 * leaves_out, cells_out (the last three may be NULL).  Row k is byte for byte what cdx_slot_prove_batch(slots[k], entropy k)
 * gives on the full slot.  A shallower slot's paths are zero-padded to max_depth.
 * A proof server gathers one period's challenges over all its slots into one call: the sampled blocks of every slot reach
 * the cell sponge together (one tile pass per source class: fake data, synthetic bytes, host memory and files), so the
 * call costs about what one slot with that many challenges costs, not the single-challenge latency once per slot.
 * n_challenges == 0 is CDX_OK and touches nothing.  CDX_ERR_ARG: a null slots, sources, entropies, indices_out or paths_out,
 * slots of different contexts, one handle with differing descriptors, a file that cannot be opened or read (bytes past
 * its end read as zeros).  CDX_ERR_SIZE: slots whose cell_size or block_size differ, sources[k].n_bytes not the slot's
 * size, more than 2^20 (challenge, sample) pairs.  CDX_ERR_STATE: a range slot, a shard or a slot without its top tree.
 * CDX_ERR_NOT_POW2: a slot whose cell count is not a power of two.  CDX_ERR_RANGE: max_depth below the deepest slot's path
 * length or above 64.  Compact and full slots may be mixed.  CDX_ERR_MISMATCH: a sampled block does not hash to its
 * retained hash; the message reads "challenge k: bytes of block N do not hash to the committed block hash", naming, among
 * the slots with a bad block, the one whose first row comes first: k is that row and N its smallest bad block (the
 * outputs are then unspecified).  Returns synchronised. */
int cdx_slots_prove_from_source(const cdx_slot* const* slots, const cdx_slot_desc* sources, const uint8_t* entropies,
                                size_t n_challenges, size_t n_samples, size_t max_depth, uint64_t* indices_out,
                                uint8_t* paths_out, uint8_t* leaves_out, uint8_t* cells_out);

/* ---- slot builder: a slot committed from blocks added in any order ------------------------------------------
 * A storage node receives a slot's blocks one at a time or in short runs, from several peers, in whatever order they
 * arrive.  A builder takes them as they come and hashes them while more arrive, so the slot is never staged whole in host
 * memory and the hashing overlaps the download.  Replaces nothing in the reference, which loads whole slots
 * (nim/slot.nim:51-73).
 *
 * cdx_slot_builder_create: the slot's shape up front, n_blocks blocks of block_size bytes; the shape rules are those of
 * cdx_slot_commit_host on n_blocks * block_size bytes (CDX_ERR_SIZE, also when that product overflows 64 bits).
 * keep_forest != 0: finish returns a full handle; keep_forest == 0: a compact one (the block forest below the block hashes
 * is never allocated, see cdx_slot_compact).  CDX_ERR_ARG for a null ctx or out, CDX_ERR_ALLOC, CDX_ERR_CUDA.
 *
 * cdx_slot_builder_add_host: blocks [first_block, first_block + n_bytes / block_size) from pageable or pinned host memory.
 * The call returns once the bytes have been copied out of `data`: the caller may reuse the buffer at once.  Statuses:
 * CDX_ERR_ARG for a null builder or data; CDX_ERR_STATE after a successful finish; CDX_ERR_SIZE when n_bytes is zero or
 * not a multiple of block_size; CDX_ERR_RANGE when the range leaves the slot (checked without overflow); CDX_ERR_STATE when
 * a block of the range has been added before (the message names the smallest such block).  A refused add changes
 * nothing.  CDX_ERR_CUDA: a device error of the tile this add completed; the builder then refuses every later call with
 * CDX_ERR_STATE.
 *
 * Tiles and memory: the bytes go through four pinned chunks of a quarter tile each into two device tiles of
 * tile_blocks = max(1, min(n_blocks, CODEX_COMMIT_TILE_MIB MiB / block_size)) blocks (256 MiB by default).  A chunk is
 * copied to the device while the next one fills; a tile is hashed when it is full, in any block order: the cell sponge,
 * the block trees in a scratch forest of the tile, and a scatter to the blocks' places in the handle, while the other
 * device tile fills.  Adds that do not complete a tile launch no kernel.  Adds of several MiB are copied by several host
 * threads, single blocks on the caller's thread.  When the pinned chunk an add needs is still in flight, the add waits for
 * it: that is the only back-pressure.  The builder's memory is fixed by the tile size, whatever the slot size (about one
 * tile of pinned host memory and two tiles plus their scratch forests on the device), besides the handle's own levels,
 * which are allocated at create.  The builder has its own streams and staging buffers: other calls on the same context,
 * and other builders, may run between two adds.
 *
 * cdx_slot_builder_finish: hashes the last partial tile, builds the slot tree and returns synchronised.  With blocks
 * missing it is CDX_ERR_STATE, the message says how many and names the smallest; the builder stays usable (add them and
 * finish again).  CDX_ERR_STATE after a successful finish, CDX_ERR_ARG for a null builder or out, CDX_ERR_CUDA.  On success
 * the handle is byte for byte what cdx_slot_commit_host on the same bytes gives (every layer, the root, the export
 * image), or with keep_forest == 0 what cdx_slot_commit_host followed by cdx_slot_compact gives (compact image,
 * cdx_slot_device_bytes).  It belongs to the builder's context, works with every call a committed slot takes and is freed
 * with cdx_slot_free; the builder's own buffers are released.  Checking the root against an expected root is the caller's
 * job (cdx_slot_root), as for cdx_slot_import.
 *
 * cdx_slot_builder_free: accepted in every state and on NULL; an unfinished slot is discarded. */
typedef struct cdx_slot_builder cdx_slot_builder;
int cdx_slot_builder_create(cdx_ctx* ctx, uint64_t n_blocks, size_t cell_size, size_t block_size, int keep_forest, cdx_slot_builder** out);
int cdx_slot_builder_add_host(cdx_slot_builder* b, uint64_t first_block, const uint8_t* data, size_t n_bytes);
int cdx_slot_builder_finish(cdx_slot_builder* b, cdx_slot** out);
void cdx_slot_builder_free(cdx_slot_builder* b);

/* ---- all GPUs of one process -------------------------------------------------------------------------------
 * For a single-process host (the Nim cli, the C++ mirror): a group owns one context and one communicator rank per
 * device and runs every collective call on one worker thread per GPU.  Results are those of rank 0. */
typedef struct cdx_group cdx_group;
/* devices == NULL or n_devices <= 0: every visible GPU */
int cdx_group_create(const int* devices, int n_devices, cdx_group** out);
void cdx_group_destroy(cdx_group* group);
int cdx_group_size(const cdx_group* group);
cdx_ctx* cdx_group_ctx(const cdx_group* group, int rank);
cdx_comm* cdx_group_comm(const cdx_group* group, int rank);
const char* cdx_group_last_error(const cdx_group* group);
/* one slot in host memory, block-range-sharded over the group's GPUs; slots_out receives cdx_group_size handles */
int cdx_group_slot_commit_host(cdx_group* group, const uint8_t* data, size_t n_bytes, size_t cell_size, size_t block_size, cdx_slot** slots_out);
int cdx_group_slot_cell_paths(cdx_group* group, cdx_slot* const* slots, const uint64_t* cell_indices, size_t n_samples, size_t max_depth,
                              uint8_t* out, uint8_t* leaf_out);
void cdx_group_slots_free(cdx_group* group, cdx_slot** slots);
/* cdx_dataset_commit / cdx_dataset_prove on every GPU of the group; datasets_out receives cdx_group_size handles */
int cdx_group_dataset_commit(cdx_group* group, const cdx_slot_desc* slots, size_t n_slots, size_t cell_size, size_t block_size,
                             int64_t keep_slot, cdx_dataset** datasets_out);
int cdx_group_dataset_prove(cdx_group* group, cdx_dataset* const* datasets, const uint8_t entropy[32], size_t n_samples, size_t max_depth,
                            uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out);
void cdx_group_datasets_free(cdx_group* group, cdx_dataset** datasets);

/* ---- sampling and data source --------------------------------------------------------------------------- */

/* indices[c-1] = low log2(n_cells) bits of sponge2([entropy, slot_root, c]), c = 1..n_samples.
 * Replaces: cellIndices / cellIndex / extractLowBits -- nim/sample/bn254.nim:16-27, nim/types/bn254.nim:47-59. */
int cdx_cell_indices(cdx_ctx* ctx, const uint8_t entropy[32], const uint8_t slot_root[32], uint64_t n_cells, size_t n_samples, uint64_t* indices);

/* The reference's fake cells [first_cell, first_cell + n_cells) into a host buffer (n_cells * cell_size bytes).
 * Replaces: slotLoadCellData(FakeData) -- nim/slot.nim:23-32,51-55. */
int cdx_fake_cells_host(cdx_ctx* ctx, uint64_t seed, uint64_t first_cell, size_t n_cells, size_t cell_size, uint8_t* out);
int cdx_fake_cells_dev(cdx_ctx* ctx, uint64_t seed, uint64_t first_cell, size_t n_cells, size_t cell_size, void* d_out, void* stream);

/* Counter-based synthetic slot bytes for benchmarks: 64-bit word i of the slot = splitmix64(seed + first_word + i)
 * (SURVEY.md section 8d config 3).  n_bytes must be a multiple of 8. */
int cdx_fill_synthetic_dev(cdx_ctx* ctx, uint64_t seed, uint64_t first_word, size_t n_bytes, void* d_out, void* stream);

/* ---- measurement ---------------------------------------------------------------------------------------- */

/* Integer-multiply roofline probe: runs a multiply stream with ILP 8 on every SM and returns the achieved rate in
 * thread-level instructions per second.  kind 0 = IMAD.WIDE.U32 without carry (each product feeds the next
 * multiplicand), 1 = IMAD.WIDE.U32.X carry chains as in the Montgomery rows, 2 = 32-bit IMAD. */
int cdx_probe_imad_rate(cdx_ctx* ctx, int kind, double* ops_per_second, double* elapsed_ms);

/* Debug aid.  With CODEX_COMMIT_GUARD=1 in the environment every device allocation of the library sits between two 4 KiB
 * guard bands that are verified when it is freed; a damaged band aborts the process with a message (the pool this was
 * developed on offers no compute-sanitizer).  This call proves the mechanism: it allocates a scoped buffer, writes one
 * byte past its end on purpose and frees it -- in guard mode the process aborts, otherwise it returns CDX_ERR_STATE
 * without touching anything. */
int cdx_debug_guard_selftest(cdx_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* CODEX_COMMIT_H */
