"""ctypes binding of the C oracle (oracle/codex_oracle.c).  TEST INFRASTRUCTURE ONLY -- see codex_oracle.h.

Field elements are python ints at this level; they cross into C as 32-byte little-endian canonical strings.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from typing import List, Optional, Sequence, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _cpu_has(*flags: str) -> bool:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    have = set(line.split(":", 1)[1].split())
                    return all(fl in have for fl in flags)
    except OSError:
        pass
    return False


_SO = os.path.join(_HERE, "build", "libcodex_oracle.so" if _cpu_has("bmi2", "adx") else "libcodex_oracle_generic.so")


def build(force: bool = False) -> str:
    """Compile the oracle with gcc (idempotent)."""
    srcs = [os.path.join(_HERE, f) for f in ("codex_oracle.c", "codex_oracle.h", "poseidon2_rc.h", "Makefile")]
    stale = force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if stale:
        subprocess.run(["make", "-C", _HERE, "-s"] + (["-B"] if force else []), check=True)
    return _SO


def use_native() -> bool:
    """Switch to a build tuned for THIS machine (-O3 -march=native), compiled here and now; used by bench.py's CPU legs so
    that the reported baseline is not handicapped by generic code.  The library goes to a fresh temporary directory
    (removed at exit), so the source tree may be read-only.  Returns False (and keeps the portable build) if the compiler
    is missing or the build fails."""
    global _SO, _lib
    out_dir = tempfile.mkdtemp(prefix="codex_oracle_native_")
    atexit.register(shutil.rmtree, out_dir, True)
    native = os.path.join(out_dir, "libcodex_oracle_native.so")
    try:
        subprocess.run(["make", "-C", _HERE, "-s", "native", "BUILD=" + out_dir], check=True, capture_output=True)
        C.CDLL(native)
    except Exception:
        return False
    _SO, _lib = native, None
    return True


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        L.orc_fr_sqr_check.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
        L.orc_fr_mul_check.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p]
        u8p, sz, u64 = C.c_char_p, C.c_size_t, C.c_uint64
        L.orc_permutation.argtypes = [u8p, u8p]
        L.orc_permutation_batch.argtypes = [u8p, u8p, sz]
        L.orc_sponge.argtypes = [u8p, sz, C.c_int, u8p]
        L.orc_bytes_to_elements.argtypes = [u8p, sz, u8p]
        L.orc_bytes_to_elements.restype = sz
        L.orc_hash_bytes.argtypes = [u8p, sz, u8p]
        L.orc_compress.argtypes = [u8p, u8p, C.c_uint32, u8p]
        L.orc_merkle_total_nodes.argtypes = [sz, C.c_int]
        L.orc_merkle_total_nodes.restype = sz
        L.orc_merkle_layers.argtypes = [u8p, sz, C.c_int, u8p]
        L.orc_merkle_root.argtypes = [u8p, sz, u8p]
        L.orc_reconstruct_root.argtypes = [u8p, u64, u64, u8p, sz, u8p]
        L.orc_gen_fake_cell.argtypes = [u64, u64, sz, u8p]
        L.orc_commit_slot.argtypes = [C.c_void_p, sz, sz, sz, C.c_int, C.c_void_p, C.c_void_p, u8p]
        L.orc_commit_fake_slot.argtypes = [u64, sz, sz, sz, C.c_int, C.c_void_p, C.c_void_p, u8p]
        L.orc_cell_index.argtypes = [u8p, u8p, u64, u64]
        L.orc_cell_index.restype = C.c_int64
        L.orc_to_decimal.argtypes = [u8p, u8p]
        _lib = L
    return _lib


def f2b(x: int) -> bytes:
    return int(x).to_bytes(32, "little")


def b2f(b: bytes) -> int:
    return int.from_bytes(b, "little")


def pack(xs: Sequence[int]) -> bytes:
    return b"".join(f2b(x) for x in xs)


def unpack(buf: bytes) -> List[int]:
    return [int.from_bytes(buf[i:i + 32], "little") for i in range(0, len(buf), 32)]


def set_use_sqr(on: bool) -> None:
    """S-box squarings through the dedicated 10-product squaring (default) or the general CIOS product; identical results"""
    lib().orc_set_use_sqr(1 if on else 0)


def have_asm() -> bool:
    return bool(lib().orc_have_asm())


def fr_mul_check(a: int, b: int) -> Tuple[int, int]:
    """(a*b mod r via the build's fast product -- MULX/ADCX/ADOX where compiled in --, via the portable C product)"""
    o1, o2 = C.create_string_buffer(32), C.create_string_buffer(32)
    lib().orc_fr_mul_check(f2b(a), f2b(b), o1, o2)
    return b2f(o1.raw), b2f(o2.raw)


def fr_sqr_check(a: int) -> Tuple[int, int]:
    """(a^2 mod r via the dedicated squaring, via the general product)"""
    o1, o2 = C.create_string_buffer(32), C.create_string_buffer(32)
    lib().orc_fr_sqr_check(f2b(a), o1, o2)
    return b2f(o1.raw), b2f(o2.raw)


def permutation(s: Sequence[int]) -> Tuple[int, int, int]:
    out = C.create_string_buffer(96)
    lib().orc_permutation(pack(s), out)
    return tuple(unpack(out.raw))


def permutation_batch_bytes(states: bytes) -> bytes:
    n = len(states) // 96
    out = C.create_string_buffer(96 * n)
    lib().orc_permutation_batch(states, out, n)
    return out.raw


def sponge(xs: Sequence[int], rate: int = 2) -> int:
    out = C.create_string_buffer(32)
    rc = lib().orc_sponge(pack(xs), len(xs), rate, out)
    if rc:
        raise ValueError(f"orc_sponge rc={rc}")
    return b2f(out.raw)


def sponge1(xs): return sponge(xs, 1)
def sponge2(xs): return sponge(xs, 2)


def bytes_to_elements(data: bytes) -> List[int]:
    out = C.create_string_buffer(32 * (len(data) // 31 + 1))
    n = lib().orc_bytes_to_elements(bytes(data), len(data), out)
    return unpack(out.raw[:32 * n])


def hash_bytes(data: bytes) -> int:
    out = C.create_string_buffer(32)
    lib().orc_hash_bytes(bytes(data), len(data), out)
    return b2f(out.raw)


def compress(x: int, y: int, key: int = 0) -> int:
    out = C.create_string_buffer(32)
    lib().orc_compress(f2b(x), f2b(y), key, out)
    return b2f(out.raw)


def merkle_layers(xs: Sequence[int], bottom: bool = True) -> List[List[int]]:
    n = len(xs)
    if n == 0:
        raise ValueError("merkle tree of empty input")
    total = lib().orc_merkle_total_nodes(n, int(bottom))
    out = C.create_string_buffer(32 * total)
    nl = lib().orc_merkle_layers(pack(xs), n, int(bottom), out)
    assert nl > 0
    flat, layers, off, m, b = unpack(out.raw), [], 0, n, bottom
    for _ in range(nl):
        layers.append(flat[off:off + m])
        off += m
        m = (m + 1) // 2
    return layers


def merkle_root(xs: Sequence[int]) -> int:
    out = C.create_string_buffer(32)
    rc = lib().orc_merkle_root(pack(xs), len(xs), out)
    if rc:
        raise ValueError("orc_merkle_root rc=%d" % rc)
    return b2f(out.raw)


def reconstruct_root(leaf: int, index: int, n_leaves: int, path: Sequence[int]) -> int:
    out = C.create_string_buffer(32)
    lib().orc_reconstruct_root(f2b(leaf), index, n_leaves, pack(path), len(path), out)
    return b2f(out.raw)


def gen_fake_cell(seed: int, idx: int, cell_size: int) -> bytes:
    out = C.create_string_buffer(cell_size)
    lib().orc_gen_fake_cell(seed & (2**64 - 1), idx, cell_size, out)
    return out.raw


def commit_slot(data, cell_size: int = 2048, block_size: int = 65536, n_threads: int = 1,
                want_cells: bool = False) -> Tuple[int, List[int], Optional[List[int]]]:
    """data: bytes-like or (address, nbytes) tuple.  Returns (root, block_hashes, cell_hashes|None)."""
    if isinstance(data, tuple):
        addr, nbytes = data
    else:
        data = bytes(data) if not isinstance(data, (bytes, bytearray)) else data
        keep = (C.c_char * len(data)).from_buffer_copy(data)
        addr, nbytes = C.addressof(keep), len(data)
    nb, ncell = nbytes // block_size, nbytes // cell_size
    bh = C.create_string_buffer(32 * nb)
    ch = C.create_string_buffer(32 * ncell) if want_cells else None
    root = C.create_string_buffer(32)
    rc = lib().orc_commit_slot(addr, nbytes, cell_size, block_size, n_threads,
                               C.addressof(ch) if ch else None, C.addressof(bh), root)
    if rc:
        raise ValueError(f"orc_commit_slot rc={rc}")
    return b2f(root.raw), unpack(bh.raw), (unpack(ch.raw) if ch else None)


def commit_fake_slot(seed: int, n_cells: int, cell_size: int = 2048, block_size: int = 65536, n_threads: int = 1,
                     want_cells: bool = False):
    k = block_size // cell_size
    bh = C.create_string_buffer(32 * (n_cells // k))
    ch = C.create_string_buffer(32 * n_cells) if want_cells else None
    root = C.create_string_buffer(32)
    rc = lib().orc_commit_fake_slot(seed & (2**64 - 1), n_cells, cell_size, block_size, n_threads,
                                    C.addressof(ch) if ch else None, C.addressof(bh), root)
    if rc:
        raise ValueError(f"orc_commit_fake_slot rc={rc}")
    return b2f(root.raw), unpack(bh.raw), (unpack(ch.raw) if ch else None)


def cell_index(entropy: int, slot_root: int, n_cells: int, counter: int) -> int:
    r = lib().orc_cell_index(f2b(entropy), f2b(slot_root), n_cells, counter)
    if r < 0:
        raise ValueError("numberOfCells is assumed to be a power of two")
    return r


def to_decimal(x: int) -> str:
    buf = C.create_string_buffer(80)
    lib().orc_to_decimal(f2b(x), buf)
    return buf.value.decode()
