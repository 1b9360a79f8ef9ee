"""Slot builder (cdx_slot_builder_*): a slot committed from blocks added in any order and in any number of pieces.

CPU part: the bookkeeping and argument checks (csrc/slot_builder.h) compiled with g++, plain and under UBSan, against a
Python restatement: ranges touching the slot's end, ranges whose end wraps 2^64, zero and non-multiple sizes, duplicates
at the start, middle and end of a range, the missing-block count and smallest index after random add sequences, adds and
finishes after a finish, and shapes whose byte count overflows.

GPU part: a builder fed as one piece, as single blocks in random order or as random runs in random order gives the handle
cdx_slot_commit_host gives (full) or commit_host + compact gives (compact): root (also against the oracle), every layer,
export image, device bytes and the answers of prove_batch / prove_from_source; slots spanning several tiles, with a tile's
sponge split over several launches; the exact launch count; the caller's buffer reused at once; every refusal with its
status and message, each followed by a correct finish; other calls and a second builder on the same context between the
adds; all of it again under CODEX_COMMIT_GUARD=1."""
import ctypes as C
import os
import random
import re
import subprocess
import sys

import pytest

from conftest import ROOT
from oracle import coracle

gpu = pytest.mark.gpu
M64 = 1 << 64
OK, ARG, SIZE, RANGE, STATE = 0, -1, -2, -4, -7

# (cell, block): cpb 1, 2, 32 and 256; 64-byte and larger multiple-of-32 cells take the TMA sponge, 36 and 100 the plain one
GEOMETRIES = [(64, 64), (36, 36), (2048, 4096), (100, 200), (2048, 65536), (36, 1152), (64, 16384), (100, 25600)]
GEOMETRY_IDS = [f"{c}x{b}" for c, b in GEOMETRIES]
SLOT_BLOCKS = (1, 2, 3, 5, 8, 33)


# ---- the bookkeeping, restated ---------------------------------------------------------------------------------

def shape_ref(n_blocks, cell, block):
    """slot_builder_shape restated with unbounded integers -> (status, message or None where only the status is pinned)"""
    n_bytes = n_blocks * block
    if n_bytes >= M64:
        return SIZE, f"slot builder: {n_blocks} blocks of {block} bytes overflow 64 bits"
    if cell == 0 or cell % 4 or cell > 1 << 30 or block == 0 or block % cell:
        return SIZE, None
    cpb = block // cell
    if cpb & (cpb - 1) or n_bytes == 0:
        return SIZE, None
    return OK, None


class BookRef:
    """slot_builder_add / _missing / _finish_status restated"""

    def __init__(self, n_blocks):
        self.n, self.added, self.finished = n_blocks, set(), False

    def add(self, first, n_bytes, block):
        if self.finished:
            return STATE, "slot builder: the slot is finished, no block can be added"
        if n_bytes == 0 or n_bytes % block:
            return SIZE, f"slot builder: an add of {n_bytes} bytes is not a non-zero multiple of the block size {block}"
        n = n_bytes // block
        if first >= self.n or n > self.n - first:
            return RANGE, f"slot builder: blocks [{first},+{n}) are outside the slot of {self.n} blocks"
        dup = [b for b in self.added if first <= b < first + n]
        if dup:
            return STATE, f"slot builder: block {min(dup)} has already been added"
        self.added.update(range(first, first + n))
        return OK, None

    def missing(self):
        miss = [b for b in range(self.n) if b not in self.added]
        return len(miss), (miss[0] if miss else self.n)

    def finish(self):
        if self.finished:
            return STATE, "slot builder: the slot is finished already"
        count, smallest = self.missing()
        if count:
            return STATE, f"slot builder: {count} of {self.n} blocks are missing, the smallest is block {smallest}"
        self.finished = True
        return OK, None


class Book:
    """the compiled bookkeeping of one builder, through tests/host_emul/slot_builder_check.cpp"""

    def __init__(self, lib, n_blocks):
        self.lib, self.h = lib, lib.book_new(n_blocks)
        self.msg = C.create_string_buffer(256)

    def add(self, first, n_bytes, block):
        n = C.c_uint64()
        self.msg.value = b""
        rc = self.lib.book_add(self.h, first, n_bytes, block, C.byref(n), self.msg, 256)
        return rc, (self.msg.value.decode() if rc else None)

    def missing(self):
        smallest = C.c_uint64()
        count = self.lib.book_missing(self.h, C.byref(smallest))
        return count, smallest.value

    def finish(self):
        self.msg.value = b""
        rc = self.lib.book_finish(self.h, self.msg, 256)
        return rc, (self.msg.value.decode() if rc else None)

    def free(self):
        self.lib.book_free(self.h)


def bind(lib):
    lib.builder_shape.restype = C.c_int
    lib.builder_shape.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_char_p, C.c_size_t]
    lib.book_new.restype = C.c_void_p
    lib.book_new.argtypes = [C.c_uint64]
    lib.book_free.argtypes = [C.c_void_p]
    lib.book_add.restype = C.c_int
    lib.book_add.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), C.c_char_p, C.c_size_t]
    lib.book_missing.restype = C.c_uint64
    lib.book_missing.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.book_finish.restype = C.c_int
    lib.book_finish.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t]
    return lib


def shape_cases():
    cases = [(4, 2048, 65536), (1, 64, 64), (33, 36, 1152), (1 << 20, 2048, 65536)]
    cases += [(n, 4, 4 << k) for n, k in (((1 << 62) - 1, 0), ((1 << 62) - 1, 2), (1 << 62, 2), ((1 << 61) + 1, 3), (M64 - 1, 0), (M64 - 1, 1))]
    cases += [(3, 0, 64), (3, 6, 12), (3, 64, 0), (3, 64, 96), (3, 64, 192), (0, 64, 64), (3, (1 << 30) + 4, (1 << 30) + 4)]
    cases += [(M64 - 1, 64, 0), ((1 << 58) + 1, 64, 64), (1 << 58, 64, 64)]
    return cases


def add_sequences():
    """(n_blocks, block, [(first, n_bytes)]) tables: edges, wraps, sizes, duplicates, then random sequences"""
    block = 64
    seqs = []
    for n in (1, 2, 63, 64, 65, 130, 1000):
        ops = [(n - 1, block), (n - 1, block), (n, block), (n - 1, 2 * block), (n, 0), (M64 - 1, block)]
        ops += [(0, n * block + block), (0, (n - 1) * block)] if n > 1 else [(0, 2 * block)]
        seqs.append((n, block, ops))
        # ranges ending exactly at the end, and one block past it
        seqs.append((n, block, [(n - k, k * block) for k in (1, 2, 3) if k <= n] + [(0, n * block), (0, (n + 1) * block)]))
    # first_block + n wrapping 2^64
    for first, nb in ((M64 - 1, 1), (M64 - 1, 2), (M64 - 3, 5), (1 << 63, (1 << 63) // block * block), (5, M64 - block), (0, M64 - block)):
        seqs.append((10, block, [(first, nb)]))
    # zero-size and non-multiple sizes
    seqs.append((10, block, [(0, 0), (0, 1), (0, block - 1), (0, block + 1), (2, 3 * block + 7), (3, M64 - 1), (3, block)]))
    # a duplicate at the start, the middle and the end of a range; two duplicates name the smaller
    for n in (10, 100, 200):
        for at in (0, n // 2, n - 1):
            ops = [(at, block)]
            ops += [(at, 3 * block)] if at + 3 <= n else []
            ops += [(max(0, at - 1), 2 * block)] if at >= 1 else []
            ops += [(max(0, at - 2), 3 * block)] if at >= 2 else []
            ops += [(0, n * block)]
            seqs.append((n, block, ops))
        seqs.append((n, block, [(n - 1, block), (3, block), (0, n * block), (4, (n - 4) * block)]))
    # runs crossing 64-block words
    seqs.append((300, block, [(63, 2 * block), (60, 10 * block), (127, 130 * block), (65, 62 * block), (0, 300 * block)]))
    # random sequences: runs of random length at random places, many refused
    rnd = random.Random(2024)
    for _ in range(60):
        n = rnd.choice((1, 7, 64, 65, 129, 500))
        ops = []
        for _ in range(rnd.randint(1, 40)):
            first = rnd.randrange(n + 2)
            ops.append((first, rnd.randint(1, max(1, n // 4)) * block))
        seqs.append((n, block, ops))
    return seqs


def run_table(lib):
    msg = C.create_string_buffer(256)
    for n_blocks, cell, block in shape_cases():
        want, want_msg = shape_ref(n_blocks, cell, block)
        got = lib.builder_shape(n_blocks % M64, cell, block, msg, 256)
        assert got == want, (n_blocks, cell, block, msg.value)
        if want_msg is not None:
            assert msg.value.decode() == want_msg
        elif want != OK:
            assert msg.value
    for n_blocks, block, ops in add_sequences():
        ref, book = BookRef(n_blocks), Book(lib, n_blocks)
        try:
            for first, nb in ops:
                assert book.add(first, nb, block) == ref.add(first, nb, block), (n_blocks, first, nb)
                assert book.missing() == ref.missing(), (n_blocks, first, nb)
            assert book.finish() == ref.finish(), n_blocks
            if ref.finished:
                assert book.add(0, block, block) == ref.add(0, block, block)
                assert book.finish() == ref.finish()
            else:                                        # the missing blocks, then a finish that succeeds
                for b in range(n_blocks):
                    if b not in ref.added:
                        assert book.add(b, block, block) == ref.add(b, block, block) == (OK, None)
                assert book.missing() == ref.missing() == (0, n_blocks)
                assert book.finish() == ref.finish() == (OK, None)
                assert book.add(n_blocks - 1, block, block) == (STATE, "slot builder: the slot is finished, no block can be added")
                assert book.finish() == (STATE, "slot builder: the slot is finished already")
        finally:
            book.free()


def test_restatement_pins_the_messages():
    ref = BookRef(10)
    assert ref.add(3, 128, 64) == (OK, None)
    assert ref.add(2, 3 * 64, 64) == (STATE, "slot builder: block 3 has already been added")
    assert ref.add(9, 128, 64) == (RANGE, "slot builder: blocks [9,+2) are outside the slot of 10 blocks")
    assert ref.add(0, 0, 64) == (SIZE, "slot builder: an add of 0 bytes is not a non-zero multiple of the block size 64")
    assert ref.finish() == (STATE, "slot builder: 8 of 10 blocks are missing, the smallest is block 0")
    assert shape_ref((1 << 62) - 1, 4, 4) == (OK, None) and shape_ref(1 << 62, 4, 4)[0] == SIZE


def _build(tmp_path_factory, name, flags):
    out = str(tmp_path_factory.mktemp(name) / f"lib{name}.so")
    src = os.path.join(ROOT, "tests", "host_emul", "slot_builder_check.cpp")
    res = subprocess.run(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-shared", "-fPIC"] + flags + ["-o", out, src],
                         capture_output=True, text=True)
    return res, out


@pytest.fixture(scope="module")
def book_lib(tmp_path_factory):
    res, out = _build(tmp_path_factory, "bookcheck", ["-O2"])
    assert res.returncode == 0, res.stderr
    return bind(C.CDLL(out))


@pytest.fixture(scope="module")
def book_lib_ubsan(tmp_path_factory):
    """the same checks built with -fsanitize=undefined -fno-sanitize-recover: any undefined behaviour on the way aborts"""
    res, out = _build(tmp_path_factory, "bookcheck_ubsan", ["-O1", "-g", "-fsanitize=undefined", "-fno-sanitize-recover=undefined"])
    if res.returncode != 0:
        pytest.skip("this g++ cannot build with -fsanitize=undefined: " + res.stderr[-200:])
    try:
        return bind(C.CDLL(out))
    except OSError as e:
        pytest.skip("the UBSan runtime is not loadable: " + str(e))


def test_bookkeeping(book_lib):
    run_table(book_lib)


def test_bookkeeping_under_ubsan(book_lib_ubsan):
    run_table(book_lib_ubsan)


# ---- GPU ------------------------------------------------------------------------------------------------------

def random_bytes(seed, n):
    import numpy as np
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8).tobytes()


def fresh_context(pkg, **env):
    """a context created with CODEX_COMMIT_* settings, which are read once per context"""
    saved = {k: os.environ.pop(k, None) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return pkg.Context(0)
    finally:
        for k, v in saved.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v


def runs(rnd, n, max_run):
    """[first, first + k) runs of random length covering 0..n-1, in random order"""
    out, b = [], 0
    while b < n:
        k = min(n - b, rnd.randint(1, max_run))
        out.append((b, k))
        b += k
    rnd.shuffle(out)
    return out


def feed(builder, data, block, order, rnd):
    n = len(data) // block
    if order == "whole":
        builder.add(0, data)
    elif order == "singles":
        for b in rnd.sample(range(n), n):
            builder.add(b, data[b * block:(b + 1) * block])
    else:
        for first, k in runs(rnd, n, max(1, n // 3)):
            builder.add(first, data[first * block:(first + k) * block])


def all_layers(slot):
    n_cells, n_blocks, bd, sd = slot.shape
    cpb = n_cells // n_blocks
    forest = [slot.read_layer(0, l, 0, n_cells if cpb == 1 else n_cells >> l) for l in range(bd + 1)]
    w, widths = n_blocks, [n_blocks]
    while len(widths) <= sd:
        w = (w + 1) // 2
        widths.append(w)
    return forest, [slot.read_layer(1, l, 0, widths[l]) for l in range(sd + 1)]


class Reference:
    """what cdx_slot_commit_host gives on `data`, before and after compaction"""

    def __init__(self, pkg, ctx, data, cell, block, entropies=(5, 1 << 200), n_samples=6):
        capi = pkg.capi
        self.desc = (capi.SRC_HOST, data, len(data))
        with ctx.slot_commit_host(data, cell, block) as s:
            self.root, self.shape = s.root, s.shape
            n_cells, _, bd, sd = s.shape
            self.md = bd + sd + 1
            self.pow2 = n_cells & (n_cells - 1) == 0
            self.layers, self.image = all_layers(s), s.export()
            self.entropies, self.n_samples = list(entropies), n_samples
            self.prove = s.prove_batch(self.entropies, n_samples, self.md) if self.pow2 else None
            s.compact()
            self.compact_image, self.compact_bytes = s.export(), s.device_bytes
            self.from_source = s.prove_from_source(self.desc, self.entropies, n_samples, self.md) if self.pow2 else None

    def check(self, slot, keep_forest, what=""):
        assert slot.root == self.root and slot.shape == self.shape, what
        if keep_forest:
            assert all_layers(slot) == self.layers, what
            assert slot.export() == self.image, what
            if self.pow2:
                assert slot.prove_batch(self.entropies, self.n_samples, self.md) == self.prove, what
        else:
            assert slot.export() == self.compact_image, what
            assert slot.device_bytes == self.compact_bytes, what
            if self.pow2:
                assert slot.prove_from_source(self.desc, self.entropies, self.n_samples, self.md) == self.from_source, what


@gpu
@pytest.mark.parametrize("cell,block", GEOMETRIES, ids=GEOMETRY_IDS)
def test_builder_equals_commit_host_and_oracle(pkg, ctx, orc, cell, block):
    rnd = random.Random(cell * 131 + block)
    for n_blocks in SLOT_BLOCKS:
        data = random_bytes(cell * block + n_blocks, n_blocks * block)
        ref = Reference(pkg, ctx, data, cell, block)
        assert ref.root == coracle.commit_slot(data, cell, block)[0], n_blocks
        for keep in (True, False):
            for order in ("whole", "singles", "runs"):
                with ctx.slot_builder(n_blocks, cell, block, keep_forest=keep) as b:
                    feed(b, data, block, order, rnd)
                    with b.finish() as s:
                        ref.check(s, keep, (n_blocks, keep, order))


@gpu
@pytest.mark.parametrize("cell,block,n_blocks", [(2048, 65536, 900), (64, 16384, 3300)], ids=["cpb32-900", "cpb256-3300"])
@pytest.mark.parametrize("max_cells", [None, 2976], ids=["one-launch", "multi-launch"])
def test_slots_spanning_several_tiles(pkg, ctx, cell, block, n_blocks, max_cells):
    """16 MiB tiles: 3.5 (cpb 32) or 3.2 (cpb 256) tiles; runs of up to 150 blocks (over the 4 MiB parallel-copy size) in random
    order straddle the four-chunk and the tile fills; with a lowered launch limit a tile's sponge takes several launches"""
    env = {"CODEX_COMMIT_TILE_MIB": 16}
    if max_cells:
        env["CODEX_COMMIT_MAX_LAUNCH_CELLS"] = max_cells
    c = fresh_context(pkg, **env)
    try:
        data = random_bytes(n_blocks + block, n_blocks * block)
        ref = Reference(pkg, c, data, cell, block)
        rnd = random.Random(n_blocks)
        for keep in (True, False):
            with c.slot_builder(n_blocks, cell, block, keep_forest=keep) as b:
                for first, k in runs(rnd, n_blocks, 150):
                    b.add(first, data[first * block:(first + k) * block])
                with b.finish() as s:
                    ref.check(s, keep, keep)
    finally:
        c.close()


def expected_launches(n_blocks, cpb, tile_blocks, max_cells, keep):
    bd = 1 if cpb == 1 else cpb.bit_length() - 1
    w, sd = n_blocks, 0
    while sd == 0 or w > 1:
        w, sd = (w + 1) // 2, sd + 1
    total = 0
    for t0 in range(0, n_blocks, tile_blocks):
        cells = min(tile_blocks, n_blocks - t0) * cpb
        total += -(-cells // max_cells) + bd + (bd + 1 if keep else 1)
    return total + sd


@gpu
def test_launch_count(pkg):
    cell, block, cpb, tile_blocks = 2048, 65536, 32, 256             # 16 MiB tiles
    c = fresh_context(pkg, CODEX_COMMIT_TILE_MIB=16)
    try:
        for n_blocks in (256, 600):
            data = random_bytes(n_blocks, n_blocks * block)
            with c.slot_commit_host(data, cell, block) as s:
                root = s.root
            for keep in (True, False):
                with c.slot_builder(n_blocks, cell, block, keep_forest=keep) as b:
                    start = c.launches
                    for i in range(tile_blocks - 1):                 # one short of a tile, block by block and in reverse
                        j = tile_blocks - 2 - i
                        b.add(j, data[j * block:(j + 1) * block])
                        assert c.launches == start, i
                    b.add(n_blocks - 1, data[(n_blocks - 1) * block:])   # completes the first tile
                    assert c.launches > start
                    rest = [j for j in range(tile_blocks - 1, n_blocks - 1)]
                    for j in rest:
                        b.add(j, data[j * block:(j + 1) * block])
                    with b.finish() as s:
                        assert c.launches - start == expected_launches(n_blocks, cpb, tile_blocks, 1 << 30, keep), (n_blocks, keep)
                        assert s.root == root
    finally:
        c.close()


@gpu
def test_caller_buffer_is_copied_before_the_add_returns(pkg):
    cell, block, n_blocks = 2048, 65536, 600
    c = fresh_context(pkg, CODEX_COMMIT_TILE_MIB=16)
    try:
        data = random_bytes(99, n_blocks * block)
        with c.slot_commit_host(data, cell, block) as s:
            root = s.root
        rnd = random.Random(3)
        for keep in (True, False):
            buf = bytearray(block)
            with c.slot_builder(n_blocks, cell, block, keep_forest=keep) as b:
                for j in rnd.sample(range(n_blocks), n_blocks):
                    buf[:] = data[j * block:(j + 1) * block]
                    b.add(j, buf)
                buf[:] = bytes(block)
                with b.finish() as s:
                    assert s.root == root
    finally:
        c.close()


def raw(ctx, call, *args):
    """-> (status, message) of one raw library call"""
    rc = getattr(ctx.lib, call)(*args)
    return rc, ctx.lib.cdx_last_error(ctx.h).decode()


@gpu
def test_refusals(pkg, ctx):
    cell, block, n_blocks = 64, 2048, 8
    data = random_bytes(7, n_blocks * block)
    with ctx.slot_commit_host(data, cell, block) as s:
        root = s.root
    blk = lambda j, k=1: data[j * block:(j + k) * block]
    out = C.c_void_p()
    lib = ctx.lib
    # null arguments
    assert lib.cdx_slot_builder_create(None, 4, cell, block, 0, C.byref(out)) == ARG
    assert raw(ctx, "cdx_slot_builder_create", ctx.h, 4, cell, block, 0, None) == (ARG, "null pointer")
    assert lib.cdx_slot_builder_add_host(None, 0, blk(0), block) == ARG
    assert lib.cdx_slot_builder_finish(None, C.byref(out)) == ARG
    lib.cdx_slot_builder_free(None)
    assert raw(ctx, "cdx_slot_builder_create", ctx.h, (1 << 62), cell, 16, 0, C.byref(out)) == \
        (SIZE, f"slot builder: {1 << 62} blocks of 16 bytes overflow 64 bits")
    assert raw(ctx, "cdx_slot_builder_create", ctx.h, 4, cell, 3 * cell, 0, C.byref(out))[0] == SIZE
    for keep in (True, False):
        with ctx.slot_builder(n_blocks, cell, block, keep_forest=keep) as b:
            h = b.h
            assert raw(ctx, "cdx_slot_builder_add_host", h, 0, None, block) == (ARG, "null pointer")
            assert raw(ctx, "cdx_slot_builder_finish", h, None) == (ARG, "null pointer")
            assert raw(ctx, "cdx_slot_builder_add_host", h, 0, blk(0), 0) == \
                (SIZE, f"slot builder: an add of 0 bytes is not a non-zero multiple of the block size {block}")
            assert raw(ctx, "cdx_slot_builder_add_host", h, 0, blk(0, 2), block + 4) == \
                (SIZE, f"slot builder: an add of {block + 4} bytes is not a non-zero multiple of the block size {block}")
            assert raw(ctx, "cdx_slot_builder_add_host", h, 7, blk(6, 2), 2 * block) == \
                (RANGE, f"slot builder: blocks [7,+2) are outside the slot of {n_blocks} blocks")
            assert raw(ctx, "cdx_slot_builder_add_host", h, M64 - 1, blk(0, 2), 2 * block) == \
                (RANGE, f"slot builder: blocks [{M64 - 1},+2) are outside the slot of {n_blocks} blocks")
            b.add(3, blk(3))
            assert raw(ctx, "cdx_slot_builder_add_host", h, 1, blk(1, 4), 4 * block) == (STATE, "slot builder: block 3 has already been added")
            assert raw(ctx, "cdx_slot_builder_finish", h, C.byref(out)) == \
                (STATE, f"slot builder: 7 of {n_blocks} blocks are missing, the smallest is block 0")
            b.add(0, blk(0, 3))                                      # the refused run left blocks 1 and 2 free
            b.add(4, blk(4, 3))
            assert raw(ctx, "cdx_slot_builder_finish", h, C.byref(out)) == \
                (STATE, f"slot builder: 1 of {n_blocks} blocks are missing, the smallest is block 7")
            b.add(7, blk(7))
            with b.finish() as s:
                assert s.root == root
            assert raw(ctx, "cdx_slot_builder_add_host", h, 0, blk(0), block) == (STATE, "slot builder: the slot is finished, no block can be added")
            assert raw(ctx, "cdx_slot_builder_finish", h, C.byref(out)) == (STATE, "slot builder: the slot is finished already")
    # freed in every state: before any add, half fed
    with ctx.slot_builder(n_blocks, cell, block) as b:
        pass
    with ctx.slot_builder(n_blocks, cell, block, keep_forest=True) as b:
        b.add(0, blk(0, 5))


@gpu
def test_context_survives_refused_calls(pkg, ctx):
    cell, block, n_blocks = 2048, 65536, 12
    data = random_bytes(12, n_blocks * block)
    ref = Reference(pkg, ctx, data, cell, block)
    with ctx.slot_builder(n_blocks, cell, block) as b:
        b.add(5, data[5 * block:6 * block])
        for k in range(100):
            kind = k % 4
            if kind == 0:
                st = raw(ctx, "cdx_slot_builder_add_host", b.h, 5, data, block)[0]
                assert st == STATE
            elif kind == 1:
                assert raw(ctx, "cdx_slot_builder_add_host", b.h, n_blocks + k, data, block)[0] == RANGE
            elif kind == 2:
                assert raw(ctx, "cdx_slot_builder_add_host", b.h, 0, data, block - 4 * k)[0] == SIZE
            else:
                assert raw(ctx, "cdx_slot_builder_finish", b.h, C.byref(C.c_void_p()))[0] == STATE
        b.add(0, data[:5 * block])
        b.add(6, data[6 * block:])
        with b.finish() as s:
            ref.check(s, False)
    with ctx.slot_commit_host(data, cell, block) as s:
        assert s.root == ref.root


@gpu
def test_other_calls_between_adds(pkg, ctx, orc):
    """commit_host of another slot, prove_from_source on a compact slot and hash_cells_dev on the builder's context, between
    its adds; and two builders fed in alternation"""
    import torch
    capi = pkg.capi
    cell, block = 2048, 65536
    c = fresh_context(pkg, CODEX_COMMIT_TILE_MIB=16)                 # the builder's tiles flush in between
    try:
        n_blocks = 300
        data = random_bytes(31, n_blocks * block)
        ref = Reference(pkg, c, data, cell, block)
        other = random_bytes(32, 8 * block)
        other_root = coracle.commit_slot(other, cell, block)[0]
        cells = random_bytes(33, 64 * cell)
        want_cells = c.hash_bytes_batch(cells, 64, cell)
        with c.slot_commit_host(other, cell, block) as comp:
            md = sum(comp.shape[2:]) + 1
            want_proof = comp.prove_batch([9, 10], 5, md)
            comp.compact()
            d_in = torch.frombuffer(bytearray(cells), dtype=torch.uint8).cuda()
            d_out = torch.zeros(32 * 64, dtype=torch.uint8, device="cuda")
            rnd = random.Random(4)
            for keep in (True, False):
                with c.slot_builder(n_blocks, cell, block, keep_forest=keep) as b:
                    for i, (first, k) in enumerate(runs(rnd, n_blocks, 40)):
                        b.add(first, data[first * block:(first + k) * block])
                        if i % 3 == 0:
                            with c.slot_commit_host(other, cell, block) as s:
                                assert s.root == other_root
                        elif i % 3 == 1:
                            assert comp.prove_from_source((capi.SRC_HOST, other, len(other)), [9, 10], 5, md)[:3] == want_proof
                        else:
                            d_out.zero_()
                            c.hash_cells_dev(d_in.data_ptr(), 64, cell, d_out.data_ptr())
                            torch.cuda.synchronize()
                            assert capi.unpack(d_out.cpu().numpy().tobytes()) == want_cells
                    with b.finish() as s:
                        ref.check(s, keep, keep)
        # two builders on one context, block by block in alternation
        data2 = random_bytes(34, n_blocks * block)
        with c.slot_commit_host(data2, cell, block) as s:
            root2 = s.root
        with c.slot_builder(n_blocks, cell, block) as b1, c.slot_builder(n_blocks, cell, block, keep_forest=True) as b2:
            order1, order2 = rnd.sample(range(n_blocks), n_blocks), rnd.sample(range(n_blocks), n_blocks)
            for j1, j2 in zip(order1, order2):
                b1.add(j1, data[j1 * block:(j1 + 1) * block])
                b2.add(j2, data2[j2 * block:(j2 + 1) * block])
            with b1.finish() as s1, b2.finish() as s2:
                assert s1.root == ref.root and s2.root == root2
    finally:
        c.close()


@gpu
def test_slot_builder_within_guard_bands():
    """every GPU test above again with CODEX_COMMIT_GUARD=1 (4 KiB bands around every device allocation of the library,
    the builder's tiles, id tables and scratch forests among them, checked when it is freed)"""
    env = dict(os.environ, CODEX_COMMIT_GUARD="1")
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-x", "-q", "-k", "not within_guard_bands",
                          "-p", "no:cacheprovider"], capture_output=True, text=True, env=env, timeout=2400, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "CODEX_COMMIT_GUARD" not in res.stderr
    assert re.search(r"\b\d+ passed", res.stdout), res.stdout[-2000:]
