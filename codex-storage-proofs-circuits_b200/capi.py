"""ctypes binding of libcodexcommit.so (include/codex_commit.h) -- the only way Python reaches the CUDA path.

There is no CPU implementation behind these calls: if the shared library is missing, or no CUDA device is
present, loading / `Context()` raises.  Field elements are python ints at this level and cross the ABI as
32-byte little-endian canonical strings (same convention as the header).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcodexcommit.so")

CDX_OK = 0
CDX_ERR_ARG, CDX_ERR_SIZE, CDX_ERR_NOT_POW2, CDX_ERR_RANGE, CDX_ERR_CUDA, CDX_ERR_ALLOC, CDX_ERR_STATE = -1, -2, -3, -4, -5, -6, -7
CDX_ERR_MISMATCH = -8

# every symbol include/codex_commit.h declares: name -> (restype, argtypes)
_vp, _u8p, _sz, _u64, _u32, _int = C.c_void_p, C.c_char_p, C.c_size_t, C.c_uint64, C.c_uint32, C.c_int
_pp = C.POINTER(C.c_void_p)
SYMBOLS = {
    "cdx_abi_version": (_int, []),
    "cdx_device_count": (_int, []),
    "cdx_ctx_create": (_int, [_int, _pp]),
    "cdx_ctx_destroy": (None, [_vp]),
    "cdx_last_error": (C.c_char_p, [_vp]),
    "cdx_status_string": (C.c_char_p, [_int]),
    "cdx_launch_count": (_u64, [_vp]),
    "cdx_ctx_stream": (_vp, [_vp]),
    "cdx_permutation_batch_host": (_int, [_vp, _vp, _vp, _sz]),
    "cdx_permutation_batch_dev": (_int, [_vp, _vp, _vp, _sz, _vp]),
    "cdx_sponge_felts_batch_host": (_int, [_vp, _vp, _sz, _sz, _int, _vp]),
    "cdx_hash_bytes_batch_host": (_int, [_vp, _vp, _sz, _sz, _vp]),
    "cdx_hash_cells_dev": (_int, [_vp, _vp, _sz, _sz, _vp, _vp]),
    "cdx_compress_batch_host": (_int, [_vp, _vp, _vp, _vp, _sz, _vp]),
    "cdx_merkle_total_nodes": (_sz, [_sz, _int]),
    "cdx_merkle_num_layers": (_int, [_sz, _int]),
    "cdx_merkle_layers_host": (_int, [_vp, _vp, _sz, _int, _vp]),
    "cdx_merkle_root_host": (_int, [_vp, _vp, _sz, _vp]),
    "cdx_slot_commit_host": (_int, [_vp, _vp, _sz, _sz, _sz, _pp]),
    "cdx_slot_commit_dev": (_int, [_vp, _vp, _sz, _sz, _sz, _vp, _pp]),
    "cdx_slot_commit_file": (_int, [_vp, C.c_char_p, _u64, _sz, _sz, _sz, _pp]),
    "cdx_slot_commit_fake": (_int, [_vp, _u64, _sz, _sz, _sz, _pp]),
    "cdx_slot_commit_range_dev": (_int, [_vp, _vp, _sz, _sz, _sz, _u64, _u64, _int, _vp, _pp]),
    "cdx_slot_commit_range_host": (_int, [_vp, _vp, _sz, _sz, _sz, _u64, _u64, _int, _pp]),
    "cdx_slot_subtree_roots_copy_dev": (_int, [_vp, _vp, _vp]),
    "cdx_slot_subtree_root_count": (_int, [_vp, C.POINTER(_u64), C.POINTER(_u64)]),
    "cdx_slot_subtree_roots_dev": (_vp, [_vp]),
    "cdx_slot_set_top_dev": (_int, [_vp, _vp, _u64, _vp]),
    "cdx_slot_export_size": (_sz, [_vp]),
    "cdx_slot_export": (_int, [_vp, _vp, _sz]),
    "cdx_slot_import": (_int, [_vp, _vp, _sz, _pp]),
    "cdx_slot_free": (None, [_vp]),
    "cdx_slot_root": (_int, [_vp, _vp]),
    "cdx_slot_shape": (_int, [_vp, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u32), C.POINTER(_u32)]),
    "cdx_slot_read_layer": (_int, [_vp, _int, _u32, _u64, _u64, _vp]),
    "cdx_slot_cell_paths": (_int, [_vp, _vp, _sz, _sz, _vp, _vp]),
    "cdx_slot_prove_batch": (_int, [_vp, _vp, _sz, _sz, _sz, _vp, _vp, _vp]),
    "cdx_reconstruct_roots_host": (_int, [_vp, _vp, _vp, _u64, _vp, _sz, _sz, _sz, _vp]),
    "cdx_cell_indices": (_int, [_vp, _vp, _vp, _u64, _sz, _vp]),
    "cdx_fake_cells_host": (_int, [_vp, _u64, _u64, _sz, _sz, _vp]),
    "cdx_fake_cells_dev": (_int, [_vp, _u64, _u64, _sz, _sz, _vp, _vp]),
    "cdx_fill_synthetic_dev": (_int, [_vp, _u64, _u64, _sz, _vp, _vp]),
    "cdx_probe_imad_rate": (_int, [_vp, _int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "cdx_debug_guard_selftest": (_int, [_vp]),
    "cdx_merkle_root_bytes_host": (_int, [_vp, _vp, _sz, _vp]),
    "cdx_slots_commit_batch_dev": (_int, [_vp, _vp, _vp, _sz, _sz, _sz, _vp, _vp]),
    "cdx_slots_commit_batch_host": (_int, [_vp, _vp, _vp, _sz, _sz, _sz, _vp]),
    "cdx_slots_commit_batch_fake": (_int, [_vp, _vp, _sz, _sz, _sz, _sz, _vp]),
    "cdx_comm_unique_id": (_int, [_vp]),
    "cdx_comm_init_rank": (_int, [_vp, _int, _int, _vp, _pp]),
    "cdx_comm_destroy": (None, [_vp]),
    "cdx_comm_rank": (_int, [_vp]),
    "cdx_comm_size": (_int, [_vp]),
    "cdx_comm_barrier": (_int, [_vp]),
    "cdx_plan_block_ranges": (_int, [_u64, _int, C.POINTER(_int), C.POINTER(_u64), C.POINTER(_u64)]),
    "cdx_block_ranges_top_level": (_int, [_u64, _int, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_int)]),
    "cdx_slot_commit_sharded_dev": (_int, [_vp, _vp, _vp, _sz, _sz, _sz, _u64, _u64, _int, _vp, _pp]),
    "cdx_slot_commit_sharded_host": (_int, [_vp, _vp, _vp, _sz, _sz, _sz, _u64, _u64, _int, _pp]),
    "cdx_slot_exchange_top": (_int, [_vp, _vp]),
    "cdx_slot_cell_paths_sharded": (_int, [_vp, _vp, _vp, _sz, _sz, _vp, _vp]),
    "cdx_slot_prove_batch_sharded": (_int, [_vp, _vp, _vp, _sz, _sz, _sz, _vp, _vp, _vp]),
    "cdx_dataset_commit": (_int, [_vp, _vp, _vp, _sz, _sz, _sz, C.c_int64, _pp]),
    "cdx_dataset_plan": (_int, [C.POINTER(_u64), _sz, _sz, _int, C.POINTER(_int)]),
    "cdx_dataset_free": (None, [_vp]),
    "cdx_dataset_root": (_int, [_vp, _vp]),
    "cdx_dataset_slot_roots": (_int, [_vp, _vp]),
    "cdx_dataset_slot_proof": (_int, [_vp, _u64, _sz, _vp]),
    "cdx_dataset_stats": (_int, [_vp, C.POINTER(_u64), C.POINTER(_u32), C.POINTER(_u32), C.POINTER(_u32)]),
    "cdx_dataset_kept_slot": (_vp, [_vp]),
    "cdx_dataset_prove": (_int, [_vp, _vp, _sz, _sz, _vp, _vp, _vp]),
    "cdx_slot_compact": (_int, [_vp]),
    "cdx_slot_device_bytes": (_sz, [_vp]),
    "cdx_slot_prove_from_source": (_int, [_vp, _vp, _vp, _sz, _sz, _sz, _vp, _vp, _vp, _vp]),
    "cdx_slots_prove_from_source": (_int, [_vp, _vp, _vp, _sz, _sz, _sz, _vp, _vp, _vp, _vp]),
    "cdx_slot_builder_create": (_int, [_vp, _u64, _sz, _sz, _int, _pp]),
    "cdx_slot_builder_add_host": (_int, [_vp, _u64, _vp, _sz]),
    "cdx_slot_builder_finish": (_int, [_vp, _pp]),
    "cdx_slot_builder_free": (None, [_vp]),
    "cdx_group_create": (_int, [C.POINTER(_int), _int, _pp]),
    "cdx_group_destroy": (None, [_vp]),
    "cdx_group_size": (_int, [_vp]),
    "cdx_group_ctx": (_vp, [_vp, _int]),
    "cdx_group_comm": (_vp, [_vp, _int]),
    "cdx_group_last_error": (C.c_char_p, [_vp]),
    "cdx_group_slot_commit_host": (_int, [_vp, _vp, _sz, _sz, _sz, _pp]),
    "cdx_group_slot_cell_paths": (_int, [_vp, _pp, _vp, _sz, _sz, _vp, _vp]),
    "cdx_group_slots_free": (None, [_vp, _pp]),
    "cdx_group_dataset_commit": (_int, [_vp, _vp, _sz, _sz, _sz, C.c_int64, _pp]),
    "cdx_group_dataset_prove": (_int, [_vp, _pp, _vp, _sz, _sz, _vp, _vp, _vp]),
    "cdx_group_datasets_free": (None, [_vp, _pp]),
}

COMM_ID_BYTES = 128
SRC_FAKE, SRC_SYNTHETIC, SRC_FILE, SRC_HOST = 0, 1, 2, 3


class SlotDesc(C.Structure):
    """cdx_slot_desc: one slot of a dataset"""
    _fields_ = [("kind", C.c_uint32), ("reserved", C.c_uint32), ("seed", C.c_uint64), ("path", C.c_char_p), ("host", C.c_void_p),
                ("n_bytes", C.c_uint64)]


def make_descs(descs):
    """[(kind, seed | path | address, n_bytes)] -> (ctypes array, keep-alive list)"""
    arr = (SlotDesc * len(descs))()
    keep = []
    for i, (kind, what, n_bytes) in enumerate(descs):
        arr[i].kind, arr[i].n_bytes = kind, n_bytes
        if kind in (SRC_FAKE, SRC_SYNTHETIC):
            arr[i].seed = int(what) & (2**64 - 1)
        elif kind == SRC_FILE:
            b = os.fsencode(what)
            keep.append(b)
            arr[i].path = b
        else:
            keep.append(what)
            arr[i].host = _addr(what)
    return arr, keep


def plan_block_ranges(n_total_blocks: int, n_ranks: int):
    """cdx_plan_block_ranges -> (top_level, [(first_block, n_blocks)] per rank)"""
    lib = load_library()
    t = C.c_int()
    first, count = (C.c_uint64 * n_ranks)(), (C.c_uint64 * n_ranks)()
    rc = lib.cdx_plan_block_ranges(n_total_blocks, n_ranks, C.byref(t), first, count)
    if rc != CDX_OK:
        raise CodexCommitError(rc, "cdx_plan_block_ranges")
    return t.value, [(int(first[r]), int(count[r])) for r in range(n_ranks)]


def block_ranges_top_level(n_total_blocks: int, ranges) -> int:
    lib = load_library()
    n = len(ranges)
    first, count = (C.c_uint64 * n)(*[r[0] for r in ranges]), (C.c_uint64 * n)(*[r[1] for r in ranges])
    t = C.c_int()
    rc = lib.cdx_block_ranges_top_level(n_total_blocks, n, first, count, C.byref(t))
    if rc != CDX_OK:
        raise CodexCommitError(rc, "cdx_block_ranges_top_level: ranges must be contiguous and cover the slot")
    return t.value


def dataset_plan(slot_bytes: Sequence[int], n_ranks: int, block_size: int = 65536) -> List[int]:
    """cdx_dataset_plan -> owner rank per slot, -1 = block-range-sharded over all ranks (no GPU needed)"""
    lib = load_library()
    n = len(slot_bytes)
    sb = (C.c_uint64 * max(n, 1))(*slot_bytes)
    owner = (C.c_int * max(n, 1))()
    rc = lib.cdx_dataset_plan(sb, n, block_size, n_ranks, owner)
    if rc != CDX_OK:
        raise CodexCommitError(rc, "cdx_dataset_plan")
    return list(owner)[:n]


def comm_unique_id() -> bytes:
    lib = load_library()
    buf = C.create_string_buffer(COMM_ID_BYTES)
    rc = lib.cdx_comm_unique_id(buf)
    if rc != CDX_OK:
        raise CodexCommitError(rc, "cdx_comm_unique_id: libnccl.so.2 could not be loaded")
    return buf.raw

_lib = None


class CodexCommitError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libcodexcommit status {status}: {message}")
        self.status = status


def load_library(path: Optional[str] = None):
    """dlopen libcodexcommit.so and bind every declared symbol; raises if the library or a symbol is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise ImportError(f"{p} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def f2b(x: int) -> bytes:
    return int(x).to_bytes(32, "little")


def b2f(b: bytes) -> int:
    return int.from_bytes(b, "little")


def pack(xs: Sequence[int]) -> bytes:
    return b"".join(int(x).to_bytes(32, "little") for x in xs)


def unpack(buf: bytes) -> List[int]:
    return [int.from_bytes(buf[i:i + 32], "little") for i in range(0, len(buf), 32)]


def _addr(buf) -> int:
    """address of a bytes / bytearray / ctypes buffer / numpy array / int (already an address)"""
    if isinstance(buf, int):
        return buf
    if isinstance(buf, bytes):           # address of the bytes object's own storage; the caller keeps it alive
        return C.cast(C.c_char_p(buf), C.c_void_p).value
    if isinstance(buf, bytearray):
        return C.addressof((C.c_char * len(buf)).from_buffer(buf))
    if hasattr(buf, "ctypes"):
        return buf.ctypes.data
    return C.addressof(buf)


def _prove_from_source_call(ctx, call, entropies, n_samples, max_depth, cell_size, cells):
    """runs call(entropies, indices, paths, leaves, cells) of one of the prove_from_source entry points on fresh output
    buffers -> (indices[k][c], paths[k][c][level], leaves[k][c], cells[k][c] = the cell's bytes, or None with cells=False)"""
    k = len(entropies)
    total = k * n_samples
    ent = b"".join(f2b(e) for e in entropies)
    idx = (C.c_uint64 * max(total, 1))()
    out = C.create_string_buffer(32 * total * max_depth if total else 1)
    leaf = C.create_string_buffer(32 * total if total else 1)
    cell = C.create_string_buffer(cell_size * total if total else 1) if cells else None
    ctx._chk(call(_addr(ent), C.addressof(idx), C.addressof(out), C.addressof(leaf), C.addressof(cell) if cells else None))
    flat = unpack(out.raw[:32 * total * max_depth])
    leaves = unpack(leaf.raw[:32 * total])
    ii = list(idx)[:total]
    paths = [flat[i * max_depth:(i + 1) * max_depth] for i in range(total)]
    raw = cell.raw if cells else None
    data = [raw[i * cell_size:(i + 1) * cell_size] if cells else None for i in range(total)]
    return ([ii[j * n_samples:(j + 1) * n_samples] for j in range(k)],
            [paths[j * n_samples:(j + 1) * n_samples] for j in range(k)],
            [leaves[j * n_samples:(j + 1) * n_samples] for j in range(k)],
            [data[j * n_samples:(j + 1) * n_samples] for j in range(k)])


class Context:
    """One per (thread, GPU): owns streams and staging buffers (cdx_ctx)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.cdx_ctx_create(device, C.byref(h))
        if rc != CDX_OK:
            raise CodexCommitError(rc, "cdx_ctx_create: " + self.lib.cdx_status_string(rc).decode() +
                                   " (a CUDA device is required; there is no CPU fallback)")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.cdx_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc: int):
        if rc != CDX_OK:
            raise CodexCommitError(rc, self.lib.cdx_last_error(self.h).decode() or self.lib.cdx_status_string(rc).decode())

    @property
    def launches(self) -> int:
        return self.lib.cdx_launch_count(self.h)

    @property
    def stream(self) -> int:
        return self.lib.cdx_ctx_stream(self.h) or 0

    # ---- hash layer ----
    def permutation_batch_bytes(self, states: bytes) -> bytes:
        n = len(states) // 96
        out = C.create_string_buffer(96 * n if n else 1)
        self._chk(self.lib.cdx_permutation_batch_host(self.h, _addr(states), C.addressof(out), n))
        return out.raw[:96 * n]

    def permutation(self, s: Sequence[int]) -> Tuple[int, int, int]:
        b = pack(s)
        return tuple(unpack(self.permutation_batch_bytes(b)))

    def permutation_batch_dev(self, d_in: int, d_out: int, n: int, stream: int = 0):
        self._chk(self.lib.cdx_permutation_batch_dev(self.h, d_in, d_out, n, stream))

    def sponge_batch(self, items: Sequence[Sequence[int]], rate: int = 2) -> List[int]:
        n = len(items)
        ln = len(items[0]) if n else 0
        assert all(len(it) == ln for it in items)
        buf = b"".join(pack(it) for it in items)
        out = C.create_string_buffer(32 * n if n else 1)
        self._chk(self.lib.cdx_sponge_felts_batch_host(self.h, _addr(buf) if buf else None, n, ln, rate, C.addressof(out)))
        return unpack(out.raw[:32 * n])

    def sponge(self, xs: Sequence[int], rate: int = 2) -> int:
        return self.sponge_batch([list(xs)], rate)[0]

    def hash_bytes_batch(self, data: bytes, n_items: int, length: int) -> List[int]:
        assert len(data) == n_items * length
        out = C.create_string_buffer(32 * n_items if n_items else 1)
        self._chk(self.lib.cdx_hash_bytes_batch_host(self.h, _addr(data) if data else None, n_items, length, C.addressof(out)))
        return unpack(out.raw[:32 * n_items])

    def hash_bytes(self, data: bytes) -> int:
        return self.hash_bytes_batch(bytes(data), 1, len(data))[0]

    def compress_batch(self, xs: Sequence[int], ys: Sequence[int], keys: Sequence[int]) -> List[int]:
        n = len(xs)
        karr = (C.c_uint32 * max(n, 1))(*keys)
        out = C.create_string_buffer(32 * n if n else 1)
        bx, by = pack(xs), pack(ys)      # named so the storage outlives the call
        self._chk(self.lib.cdx_compress_batch_host(self.h, _addr(bx), _addr(by), C.addressof(karr), n, C.addressof(out)))
        return unpack(out.raw[:32 * n])

    def compress(self, x: int, y: int, key: int = 0) -> int:
        return self.compress_batch([x], [y], [key])[0]

    # ---- Merkle ----
    def merkle_layers(self, leaves: Sequence[int], bottom: bool = True) -> List[List[int]]:
        n = len(leaves)
        total = self.lib.cdx_merkle_total_nodes(n, int(bottom))
        out = C.create_string_buffer(32 * total if total else 1)
        bl = pack(leaves)
        self._chk(self.lib.cdx_merkle_layers_host(self.h, _addr(bl) if n else None, n, int(bottom), C.addressof(out)))
        flat, layers, off, m = unpack(out.raw[:32 * total]), [], 0, n
        for _ in range(self.lib.cdx_merkle_num_layers(n, int(bottom))):
            layers.append(flat[off:off + m])
            off += m
            m = (m + 1) // 2
        return layers

    def merkle_root(self, leaves: Sequence[int]) -> int:
        out = C.create_string_buffer(32)
        n = len(leaves)
        bl = pack(leaves)
        self._chk(self.lib.cdx_merkle_root_host(self.h, _addr(bl) if n else None, n, out))
        return b2f(out.raw)

    def merkle_root_bytes(self, data: bytes) -> int:
        """Merkle.digest(openArray[byte]) -- testvectors.nim:60-66"""
        out = C.create_string_buffer(32)
        d = bytes(data)
        self._chk(self.lib.cdx_merkle_root_bytes_host(self.h, _addr(d) if d else None, len(d), out))
        return b2f(out.raw)

    # ---- many small slots ----
    def slots_commit_batch_host(self, data, slot_bytes: Sequence[int], cell_size: int = 2048, block_size: int = 65536) -> List[int]:
        n = len(slot_bytes)
        sb = (C.c_uint64 * max(n, 1))(*slot_bytes)
        out = C.create_string_buffer(32 * n if n else 1)
        self._chk(self.lib.cdx_slots_commit_batch_host(self.h, _addr(data), sb, n, cell_size, block_size, out))
        return unpack(out.raw[:32 * n])

    def slots_commit_batch_dev(self, d_data: int, slot_bytes: Sequence[int], cell_size: int = 2048, block_size: int = 65536, stream: int = 0) -> List[int]:
        n = len(slot_bytes)
        sb = (C.c_uint64 * max(n, 1))(*slot_bytes)
        out = C.create_string_buffer(32 * n if n else 1)
        self._chk(self.lib.cdx_slots_commit_batch_dev(self.h, d_data, sb, n, cell_size, block_size, stream, out))
        return unpack(out.raw[:32 * n])

    def slots_commit_batch_fake(self, seeds: Sequence[int], n_cells: int, cell_size: int = 2048, block_size: int = 65536) -> List[int]:
        n = len(seeds)
        sd = (C.c_uint64 * max(n, 1))(*[x & (2**64 - 1) for x in seeds])
        out = C.create_string_buffer(32 * n if n else 1)
        self._chk(self.lib.cdx_slots_commit_batch_fake(self.h, sd, n, n_cells, cell_size, block_size, out))
        return unpack(out.raw[:32 * n])

    # ---- several GPUs ----
    def comm_init(self, n_ranks: int, rank: int, unique_id: Optional[bytes]) -> "Comm":
        h = C.c_void_p()
        self._chk(self.lib.cdx_comm_init_rank(self.h, n_ranks, rank, unique_id, C.byref(h)))
        return Comm(self, h)

    def slot_commit_sharded_dev(self, comm: "Comm", d_data: int, n_local_bytes: int, cell_size: int, block_size: int, first_block: int,
                                n_total_blocks: int, top_level: int, stream: int = 0) -> "Slot":
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_commit_sharded_dev(self.h, comm.h if comm else None, d_data, n_local_bytes, cell_size, block_size, first_block,
                                                       n_total_blocks, top_level, stream, C.byref(h)))
        return Slot(self, h)

    def slot_commit_sharded_host(self, comm: "Comm", data, n_local_bytes: int, cell_size: int, block_size: int, first_block: int,
                                 n_total_blocks: int, top_level: int) -> "Slot":
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_commit_sharded_host(self.h, comm.h if comm else None, _addr(data) if n_local_bytes else None, n_local_bytes,
                                                        cell_size, block_size, first_block, n_total_blocks, top_level, C.byref(h)))
        return Slot(self, h)

    def dataset_commit(self, comm: Optional["Comm"], descs, cell_size: int = 2048, block_size: int = 65536, keep_slot: int = -1) -> "Dataset":
        """descs: [(kind, seed | path | buffer, n_bytes)]"""
        arr, keep = make_descs(descs)
        h = C.c_void_p()
        self._chk(self.lib.cdx_dataset_commit(self.h, comm.h if comm else None, arr, len(descs), cell_size, block_size, keep_slot, C.byref(h)))
        return Dataset(self, h, len(descs))

    # ---- slots ----
    def slot_commit_host(self, data, cell_size: int = 2048, block_size: int = 65536, n_bytes: Optional[int] = None) -> "Slot":
        nb = n_bytes if n_bytes is not None else (data.nbytes if hasattr(data, "nbytes") else len(data))
        h = C.c_void_p()
        keep = data                      # keep the buffer alive for the duration of the call
        self._chk(self.lib.cdx_slot_commit_host(self.h, _addr(keep), nb, cell_size, block_size, C.byref(h)))
        return Slot(self, h)

    def slot_commit_dev(self, d_data: int, n_bytes: int, cell_size: int = 2048, block_size: int = 65536, stream: int = 0) -> "Slot":
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_commit_dev(self.h, d_data, n_bytes, cell_size, block_size, stream, C.byref(h)))
        return Slot(self, h)

    def slot_commit_file(self, path: str, n_bytes: int, offset: int = 0, cell_size: int = 2048, block_size: int = 65536) -> "Slot":
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_commit_file(self.h, os.fsencode(path), offset, n_bytes, cell_size, block_size, C.byref(h)))
        return Slot(self, h)

    def slot_builder(self, n_blocks: int, cell_size: int = 2048, block_size: int = 65536, keep_forest: bool = False) -> "SlotBuilder":
        """a slot of n_blocks blocks committed from blocks added in any order (cdx_slot_builder_create); finish() returns a
        full handle with keep_forest, else a compact one"""
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_builder_create(self.h, n_blocks, cell_size, block_size, int(bool(keep_forest)), C.byref(h)))
        return SlotBuilder(self, h, block_size)

    def slot_import(self, image: bytes) -> "Slot":
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_import(self.h, _addr(image), len(image), C.byref(h)))
        return Slot(self, h)

    def slot_commit_fake(self, seed: int, n_cells: int, cell_size: int = 2048, block_size: int = 65536) -> "Slot":
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_commit_fake(self.h, seed & (2**64 - 1), n_cells, cell_size, block_size, C.byref(h)))
        return Slot(self, h)

    def slot_commit_range_dev(self, d_data: int, n_local_bytes: int, cell_size: int, block_size: int, first_block: int,
                              n_total_blocks: int, top_level: int, stream: int = 0) -> "Slot":
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_commit_range_dev(self.h, d_data, n_local_bytes, cell_size, block_size, first_block,
                                                     n_total_blocks, top_level, stream, C.byref(h)))
        return Slot(self, h)

    def slot_commit_range_host(self, data, cell_size: int, block_size: int, first_block: int, n_total_blocks: int,
                               top_level: int, n_bytes: Optional[int] = None) -> "Slot":
        nb = n_bytes if n_bytes is not None else (data.nbytes if hasattr(data, "nbytes") else len(data))
        h = C.c_void_p()
        self._chk(self.lib.cdx_slot_commit_range_host(self.h, _addr(data), nb, cell_size, block_size, first_block,
                                                      n_total_blocks, top_level, C.byref(h)))
        return Slot(self, h)

    def hash_cells_dev(self, d_data: int, n_cells: int, cell_size: int, d_out: int, stream: int = 0):
        self._chk(self.lib.cdx_hash_cells_dev(self.h, d_data, n_cells, cell_size, d_out, stream))

    def reconstruct_roots(self, leaves: Sequence[int], indices: Sequence[int], n_leaves: int, paths: Sequence[Sequence[int]],
                          depth: Optional[int] = None) -> List[int]:
        """batched reconstructRoot (merkle.nim:51-74): one root per (leaf, index, path)"""
        n = len(leaves)
        stride = len(paths[0]) if n else 0
        depth = stride if depth is None else depth
        bl, bp = pack(leaves), b"".join(pack(p) for p in paths)
        idx = (C.c_uint64 * max(n, 1))(*indices)
        out = C.create_string_buffer(32 * n if n else 1)
        self._chk(self.lib.cdx_reconstruct_roots_host(self.h, _addr(bl) if n else None, C.addressof(idx), n_leaves,
                                                      _addr(bp) if bp else None, stride, depth, n, C.addressof(out)))
        return unpack(out.raw[:32 * n])

    # ---- sampling / data ----
    def cell_indices(self, entropy: int, slot_root: int, n_cells: int, n_samples: int) -> List[int]:
        out = (C.c_uint64 * max(n_samples, 1))()
        be, br = f2b(entropy), f2b(slot_root)
        self._chk(self.lib.cdx_cell_indices(self.h, _addr(be), _addr(br), n_cells, n_samples, C.addressof(out)))
        return list(out)[:n_samples]

    def fake_cells(self, seed: int, first_cell: int, n_cells: int, cell_size: int) -> bytes:
        out = C.create_string_buffer(n_cells * cell_size if n_cells else 1)
        self._chk(self.lib.cdx_fake_cells_host(self.h, seed & (2**64 - 1), first_cell, n_cells, cell_size, C.addressof(out)))
        return out.raw[:n_cells * cell_size]

    def fake_cells_dev(self, seed: int, first_cell: int, n_cells: int, cell_size: int, d_out: int, stream: int = 0):
        self._chk(self.lib.cdx_fake_cells_dev(self.h, seed & (2**64 - 1), first_cell, n_cells, cell_size, d_out, stream))

    def fill_synthetic_dev(self, seed: int, first_word: int, n_bytes: int, d_out: int, stream: int = 0):
        self._chk(self.lib.cdx_fill_synthetic_dev(self.h, seed & (2**64 - 1), first_word, n_bytes, d_out, stream))

    # ---- compact commitments ----
    def prove_from_sources(self, rows, n_samples: int, max_depth: int, cells: bool = True):
        """Slot.prove_from_source over many slots in one call (cdx_slots_prove_from_source).  rows: [(slot, desc, entropy)],
        desc a (kind, seed | path | buffer, n_bytes) tuple as make_descs takes; a slot may appear in several rows, with
        equal descriptors.  -> (indices[k][c], paths[k][c][level], leaves[k][c], cells[k][c]), row k answering its own slot"""
        arr, keep = make_descs([d for _, d, _ in rows])
        handles = (C.c_void_p * max(len(rows), 1))(*[s.h for s, _, _ in rows])
        cell_size = rows[0][1][2] // rows[0][0].shape[0] if rows else 0
        call = lambda ent, idx, out, leaf, cell: self.lib.cdx_slots_prove_from_source(handles, arr, ent, len(rows), n_samples, max_depth,
                                                                                      idx, out, leaf, cell)
        res = _prove_from_source_call(self, call, [e for _, _, e in rows], n_samples, max_depth, cell_size, cells)
        del keep
        return res

    def probe_imad_rate(self, kind: int = 0) -> Tuple[float, float]:
        ops, ms = C.c_double(), C.c_double()
        self._chk(self.lib.cdx_probe_imad_rate(self.h, kind, C.byref(ops), C.byref(ms)))
        return ops.value, ms.value


class Slot:
    """A committed slot: all Merkle layers resident in HBM (cdx_slot)."""

    def __init__(self, ctx: Context, h):
        self.ctx, self.h = ctx, h

    def free(self):
        if getattr(self, "h", None):
            self.ctx.lib.cdx_slot_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.free()

    @property
    def root(self) -> int:
        out = C.create_string_buffer(32)
        self.ctx._chk(self.ctx.lib.cdx_slot_root(self.h, out))
        return b2f(out.raw)

    @property
    def shape(self):
        nc, nb, bd, sd = C.c_uint64(), C.c_uint64(), C.c_uint32(), C.c_uint32()
        self.ctx._chk(self.ctx.lib.cdx_slot_shape(self.h, C.byref(nc), C.byref(nb), C.byref(bd), C.byref(sd)))
        return nc.value, nb.value, bd.value, sd.value

    def read_layer(self, tree: int, level: int, first: int, count: int) -> List[int]:
        out = C.create_string_buffer(32 * count if count else 1)
        self.ctx._chk(self.ctx.lib.cdx_slot_read_layer(self.h, tree, level, first, count, C.addressof(out)))
        return unpack(out.raw[:32 * count])

    def cell_paths(self, cell_indices: Sequence[int], max_depth: int):
        """-> (paths[n][max_depth], leaves[n])"""
        n = len(cell_indices)
        idx = (C.c_uint64 * max(n, 1))(*cell_indices)
        out = C.create_string_buffer(32 * n * max_depth if n else 1)
        leaf = C.create_string_buffer(32 * n if n else 1)
        self.ctx._chk(self.ctx.lib.cdx_slot_cell_paths(self.h, C.addressof(idx), n, max_depth, C.addressof(out), C.addressof(leaf)))
        flat = unpack(out.raw[:32 * n * max_depth])
        return [flat[i * max_depth:(i + 1) * max_depth] for i in range(n)], unpack(leaf.raw[:32 * n])

    def prove_batch(self, entropies: Sequence[int], n_samples: int, max_depth: int):
        """answer many challenges at once: -> (indices[k][c], paths[k][c][level], leaves[k][c])"""
        k = len(entropies)
        total = k * n_samples
        ent = b"".join(f2b(e) for e in entropies)
        idx = (C.c_uint64 * max(total, 1))()
        out = C.create_string_buffer(32 * total * max_depth if total else 1)
        leaf = C.create_string_buffer(32 * total if total else 1)
        self.ctx._chk(self.ctx.lib.cdx_slot_prove_batch(self.h, _addr(ent), k, n_samples, max_depth, C.addressof(idx), C.addressof(out),
                                                        C.addressof(leaf)))
        flat = unpack(out.raw[:32 * total * max_depth])
        leaves = unpack(leaf.raw[:32 * total])
        ii = list(idx)[:total]
        paths = [flat[i * max_depth:(i + 1) * max_depth] for i in range(total)]
        return ([ii[j * n_samples:(j + 1) * n_samples] for j in range(k)],
                [paths[j * n_samples:(j + 1) * n_samples] for j in range(k)],
                [leaves[j * n_samples:(j + 1) * n_samples] for j in range(k)])

    def compact(self):
        """release the block forest below the block hashes (cdx_slot_compact); answer challenges with prove_from_source"""
        self.ctx._chk(self.ctx.lib.cdx_slot_compact(self.h))

    @property
    def device_bytes(self) -> int:
        """device memory the handle holds for its tree levels"""
        return self.ctx.lib.cdx_slot_device_bytes(self.h)

    def prove_from_source(self, desc, entropies: Sequence[int], n_samples: int, max_depth: int, cells: bool = True):
        """prove_batch from the slot's bytes, re-hashing only the sampled blocks (works on a compact slot).
        desc: one (kind, seed | path | buffer, n_bytes) tuple as make_descs takes.
        -> (indices[k][c], paths[k][c][level], leaves[k][c], cells[k][c] = the cell's bytes, or None with cells=False)"""
        arr, keep = make_descs([desc])
        cell_size = desc[2] // self.shape[0]          # the call fails with CDX_ERR_SIZE before writing if n_bytes is not the slot size
        call = lambda ent, idx, out, leaf, cell: self.ctx.lib.cdx_slot_prove_from_source(self.h, arr, ent, len(entropies), n_samples, max_depth,
                                                                                         idx, out, leaf, cell)
        res = _prove_from_source_call(self.ctx, call, entropies, n_samples, max_depth, cell_size, cells)
        del keep
        return res

    def export(self) -> bytes:
        n = self.ctx.lib.cdx_slot_export_size(self.h)
        if n == 0:
            raise CodexCommitError(CDX_ERR_STATE, "only whole slots with their top tree can be exported")
        buf = C.create_string_buffer(n)
        self.ctx._chk(self.ctx.lib.cdx_slot_export(self.h, C.addressof(buf), n))
        return buf.raw

    def subtree_roots(self):
        first, cnt = C.c_uint64(), C.c_uint64()
        self.ctx._chk(self.ctx.lib.cdx_slot_subtree_root_count(self.h, C.byref(first), C.byref(cnt)))
        return first.value, cnt.value, (self.ctx.lib.cdx_slot_subtree_roots_dev(self.h) or 0)

    def subtree_roots_copy_dev(self, d_dst: int, stream: int = 0):
        self.ctx._chk(self.ctx.lib.cdx_slot_subtree_roots_copy_dev(self.h, d_dst, stream))

    def set_top_dev(self, d_nodes: int, n_nodes: int, stream: int = 0):
        self.ctx._chk(self.ctx.lib.cdx_slot_set_top_dev(self.h, d_nodes, n_nodes, stream))

    def exchange_top(self, comm: Optional["Comm"]):
        self.ctx._chk(self.ctx.lib.cdx_slot_exchange_top(self.h, comm.h if comm else None))

    def cell_paths_sharded(self, comm: Optional["Comm"], cell_indices: Sequence[int], max_depth: int):
        """collective: every rank receives (paths[n][max_depth], leaves[n])"""
        n = len(cell_indices)
        idx = (C.c_uint64 * max(n, 1))(*cell_indices)
        out = C.create_string_buffer(32 * n * max_depth if n else 1)
        leaf = C.create_string_buffer(32 * n if n else 1)
        self.ctx._chk(self.ctx.lib.cdx_slot_cell_paths_sharded(self.h, comm.h if comm else None, C.addressof(idx), n, max_depth, C.addressof(out),
                                                               C.addressof(leaf)))
        flat = unpack(out.raw[:32 * n * max_depth])
        return [flat[i * max_depth:(i + 1) * max_depth] for i in range(n)], unpack(leaf.raw[:32 * n])

    def prove_batch_sharded(self, comm: Optional["Comm"], entropies: Sequence[int], n_samples: int, max_depth: int):
        k = len(entropies)
        total = k * n_samples
        ent = b"".join(f2b(e) for e in entropies)
        idx = (C.c_uint64 * max(total, 1))()
        out = C.create_string_buffer(32 * total * max_depth if total else 1)
        leaf = C.create_string_buffer(32 * total if total else 1)
        self.ctx._chk(self.ctx.lib.cdx_slot_prove_batch_sharded(self.h, comm.h if comm else None, _addr(ent), k, n_samples, max_depth, C.addressof(idx),
                                                                C.addressof(out), C.addressof(leaf)))
        flat = unpack(out.raw[:32 * total * max_depth])
        leaves = unpack(leaf.raw[:32 * total])
        ii = list(idx)[:total]
        paths = [flat[i * max_depth:(i + 1) * max_depth] for i in range(total)]
        return ([ii[j * n_samples:(j + 1) * n_samples] for j in range(k)],
                [paths[j * n_samples:(j + 1) * n_samples] for j in range(k)],
                [leaves[j * n_samples:(j + 1) * n_samples] for j in range(k)])


class SlotBuilder:
    """A slot being committed from blocks added in any order and in any number of pieces (cdx_slot_builder)."""

    def __init__(self, ctx: Context, h, block_size: int):
        self.ctx, self.h, self.block_size = ctx, h, block_size

    def add(self, first_block: int, data, n_bytes: Optional[int] = None):
        """blocks [first_block, first_block + n_bytes / block_size) from `data` (what _addr takes); the buffer may be reused
        as soon as the call returns"""
        nb = n_bytes if n_bytes is not None else (data.nbytes if hasattr(data, "nbytes") else len(data))
        keep = data                      # keep the buffer alive for the duration of the call
        self.ctx._chk(self.ctx.lib.cdx_slot_builder_add_host(self.h, first_block, _addr(keep), nb))

    def finish(self) -> Slot:
        """the committed slot; raises (and stays usable) while blocks are missing"""
        h = C.c_void_p()
        self.ctx._chk(self.ctx.lib.cdx_slot_builder_finish(self.h, C.byref(h)))
        return Slot(self.ctx, h)

    def free(self):
        if getattr(self, "h", None):
            self.ctx.lib.cdx_slot_builder_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.free()


class Comm:
    """One rank of a communicator (cdx_comm): NCCL inside the library, nothing for a single rank."""

    def __init__(self, ctx: Context, h):
        self.ctx, self.h = ctx, h

    @property
    def rank(self) -> int:
        return self.ctx.lib.cdx_comm_rank(self.h)

    @property
    def size(self) -> int:
        return self.ctx.lib.cdx_comm_size(self.h)

    def barrier(self):
        self.ctx._chk(self.ctx.lib.cdx_comm_barrier(self.h))

    def destroy(self):
        if getattr(self, "h", None):
            self.ctx.lib.cdx_comm_destroy(self.h)
            self.h = None


class Dataset:
    """A committed dataset (cdx_dataset): slot roots, dataset tree, optionally one retained slot."""

    def __init__(self, ctx: Context, h, n_slots: int):
        self.ctx, self.h, self.n_slots = ctx, h, n_slots

    def free(self):
        if getattr(self, "h", None):
            self.ctx.lib.cdx_dataset_free(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.free()

    @property
    def root(self) -> int:
        out = C.create_string_buffer(32)
        self.ctx._chk(self.ctx.lib.cdx_dataset_root(self.h, out))
        return b2f(out.raw)

    @property
    def slot_roots(self) -> List[int]:
        out = C.create_string_buffer(32 * self.n_slots)
        self.ctx._chk(self.ctx.lib.cdx_dataset_slot_roots(self.h, out))
        return unpack(out.raw)

    def slot_proof(self, slot_index: int, max_log2_nslots: int) -> List[int]:
        out = C.create_string_buffer(32 * max_log2_nslots if max_log2_nslots else 1)
        self.ctx._chk(self.ctx.lib.cdx_dataset_slot_proof(self.h, slot_index, max_log2_nslots, out))
        return unpack(out.raw[:32 * max_log2_nslots])

    @property
    def stats(self):
        b, w, ba, sh = C.c_uint64(), C.c_uint32(), C.c_uint32(), C.c_uint32()
        self.ctx._chk(self.ctx.lib.cdx_dataset_stats(self.h, C.byref(b), C.byref(w), C.byref(ba), C.byref(sh)))
        return {"bytes_local": b.value, "whole": w.value, "batched": ba.value, "sharded": sh.value}

    def prove(self, entropy: int, n_samples: int, max_depth: int):
        """-> (indices[n], paths[n][max_depth], leaves[n]); collective if the dataset has a communicator"""
        idx = (C.c_uint64 * max(n_samples, 1))()
        out = C.create_string_buffer(32 * n_samples * max_depth if n_samples else 1)
        leaf = C.create_string_buffer(32 * n_samples if n_samples else 1)
        be = f2b(entropy)
        self.ctx._chk(self.ctx.lib.cdx_dataset_prove(self.h, _addr(be), n_samples, max_depth, idx, out, leaf))
        flat = unpack(out.raw[:32 * n_samples * max_depth])
        return (list(idx)[:n_samples], [flat[i * max_depth:(i + 1) * max_depth] for i in range(n_samples)], unpack(leaf.raw[:32 * n_samples]))
