"""Compact commitments, many slots in one call: cdx_slots_prove_from_source answers each challenge row against its own slot,
re-hashing every sampled (slot, block) pair once.

Every row must be byte for byte what cdx_slot_prove_batch gave on its slot before compaction, at cells-per-block 1, 2, 32
and 256, on the TMA and the plain-load cell sponge, with every source kind and with compact and full slots of different
depths mixed; cells must be the source bytes; each slot's first row must match the oracle's paths, and every row must
reconstruct its own slot's root in two stages.  Also: rows that all name one slot give exactly the one-slot call, the
launch count of hundreds of slots does not depend on their number, which slot and block a mismatch names, every refused
argument, and all of it again under CODEX_COMMIT_GUARD=1."""
import ctypes as C
import os
import random
import re
import subprocess
import sys

import pytest

from conftest import ROOT
from oracle import coracle, pyoracle

gpu = pytest.mark.gpu
R = 21888242871839275222246405745257275088548364400416034343698204186575808495617

# (cell, block): cpb 1, 2, 32 and 256; 64-byte and larger multiple-of-32 cells take the TMA sponge, 36 and 100 the plain one
GEOMETRIES = [(64, 64), (36, 36), (2048, 4096), (100, 200), (2048, 65536), (36, 1152), (64, 16384), (100, 25600)]
GEOMETRY_IDS = [f"{c}x{b}" for c, b in GEOMETRIES]


@pytest.fixture(scope="module", autouse=True)
def c_primitives(orc):
    pyoracle.use_c_primitives(True)
    yield
    pyoracle.use_c_primitives(False)


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


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


def synthetic_ref(seed, n):
    """the first n bytes of a synthetic slot: byte b is byte b % 8 of splitmix64(seed + b / 8), little-endian"""
    import bench
    return bench.synthetic_bytes_host(seed, 0, (n + 7) // 8 * 8)[:n].tobytes()


def random_bytes(seed, n):
    import numpy as np
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8)


class Expected:
    """the oracle's slot over `data`: block trees, slot tree and the merged, padded path of any cell"""

    def __init__(self, data, cell, block):
        self.cpb = block // cell
        self.root, bh, ch = coracle.commit_slot(bytes(data), cell, block, want_cells=True)
        self.trees = [coracle.merkle_layers(ch[b * self.cpb:(b + 1) * self.cpb]) for b in range(len(bh))]
        self.slot = coracle.merkle_layers(bh)

    def path(self, i, max_depth):
        merged = pyoracle.merge_merkle_proofs(pyoracle.merkle_proof(self.trees[i // self.cpb], i % self.cpb),
                                              pyoracle.merkle_proof(self.slot, i // self.cpb))
        return pyoracle.pad_merkle_proof(merged, max_depth).merkle_path, merged.leaf_value


def two_stage_roots(ctx, slot, idx, paths, leaves):
    """the verifier's view (Slot.hs:189-217) of one row: block trees from the leaves, then the slot tree from the block hashes"""
    n_cells, n_blocks, bd, sd = slot.shape
    cpb = n_cells // n_blocks
    blk = ctx.reconstruct_roots(leaves, [i % cpb for i in idx], cpb, paths, bd)
    return ctx.reconstruct_roots(blk, [i // cpb for i in idx], n_blocks, [p[bd:] for p in paths], sd)


def expect_error(pkg, status, call, message=None):
    with pytest.raises(pkg.CodexCommitError) as e:
        call()
    assert e.value.status == status, str(e.value)
    if message:
        assert message in str(e.value), str(e.value)


class SlotSet:
    """slots committed from the four source kinds: .slots[name] = (slot, desc, data bytes)"""

    def __init__(self, pkg, ctx, torch, tmp_path, cell, block):
        self.capi, self.ctx, self.cell, self.block = pkg.capi, ctx, cell, block
        self.slots, self.bufs = {}, []
        self.torch, self.tmp_path = torch, tmp_path

    def fake(self, name, seed, n_blocks):
        n_cells = n_blocks * self.block // self.cell
        data = self.ctx.fake_cells(seed, 0, n_cells, self.cell)
        self.slots[name] = (self.ctx.slot_commit_fake(seed, n_cells, self.cell, self.block), (self.capi.SRC_FAKE, seed, len(data)), data)

    def synthetic(self, name, seed, n_blocks):
        n = n_blocks * self.block
        d = self.torch.empty(n, dtype=self.torch.uint8, device="cuda")
        self.ctx.fill_synthetic_dev(seed, 0, n, d.data_ptr())
        self.torch.cuda.synchronize()
        slot = self.ctx.slot_commit_dev(d.data_ptr(), n, self.cell, self.block)
        self.torch.cuda.synchronize()
        self.bufs.append(d)
        self.slots[name] = (slot, (self.capi.SRC_SYNTHETIC, seed, n), synthetic_ref(seed, n))

    def host(self, name, seed, n_blocks):
        host = random_bytes(seed, n_blocks * self.block)
        self.bufs.append(host)
        self.slots[name] = (self.ctx.slot_commit_host(host, self.cell, self.block), (self.capi.SRC_HOST, host, host.size), host.tobytes())

    def file(self, name, seed, n_blocks):
        host = random_bytes(seed, n_blocks * self.block)
        path = str(self.tmp_path / f"{name}.dat")
        host.tofile(path)
        self.slots[name] = (self.ctx.slot_commit_file(path, host.size, 0, self.cell, self.block), (self.capi.SRC_FILE, path, host.size), host.tobytes())

    def free(self):
        for slot, _, _ in self.slots.values():
            slot.free()


def check_rows(ctx, rows, got, want, data, n_samples, md, cell):
    """row k of `got` equals want[k] (prove_batch of its slot), its cells are data[k]'s bytes and it reconstructs its root"""
    idx, paths, leaves, cells = got
    assert len(idx) == len(rows)
    for k, (slot, _, _) in enumerate(rows):
        assert (idx[k], paths[k], leaves[k]) == want[k], k
        for i, c in zip(idx[k], cells[k]):
            assert c == bytes(data[k][i * cell:(i + 1) * cell]), (k, i)
        assert two_stage_roots(ctx, slot, idx[k], paths[k], leaves[k]) == [slot.root] * n_samples, k


# ---- equality with the full slots, at every geometry ------------------------------------------------------------

@gpu
@pytest.mark.parametrize("cell,block", GEOMETRIES, ids=GEOMETRY_IDS)
def test_many_slots_equal_full_slots(pkg, ctx, torch_mod, tmp_path, cell, block):
    """six slots of 1 to 16 blocks (slot depth 0 beside depth 4), every source kind, compact and full handles mixed; rows
    interleaved across slots, one slot in several rows, one row repeated"""
    ss = SlotSet(pkg, ctx, torch_mod, tmp_path, cell, block)
    base = 7919 * cell + block
    ss.fake("a", base + 1, 1)
    ss.synthetic("b", base + 2, 2)
    ss.host("c", base + 3, 4)
    ss.file("d", base + 4, 8)
    ss.fake("e", base + 5, 16)
    ss.synthetic("f", base + 6, 16)
    try:
        rnd = random.Random(base)
        ent = [0, 1, R - 1] + [rnd.getrandbits(254) % R for _ in range(8)]
        plan = [("a", 0), ("b", 1), ("c", 2), ("a", 3), ("d", 4), ("e", 5), ("f", 6), ("c", 7), ("b", 1), ("e", 8), ("d", 9), ("a", 10)]
        rows = [(ss.slots[n][0], ss.slots[n][1], ent[e]) for n, e in plan]
        data = [ss.slots[n][2] for n, _ in plan]
        bd = ss.slots["a"][0].shape[2]
        md = bd + max(s.shape[3] for s, _, _ in ss.slots.values()) + 2
        n_samples = 12
        want = [slot.prove_batch([e], n_samples, md) for slot, _, e in rows]
        want = [(w[0][0], w[1][0], w[2][0]) for w in want]
        for n in ("a", "c", "d", "f"):
            ss.slots[n][0].compact()
        got = ctx.prove_from_sources(rows, n_samples, md)
        check_rows(ctx, rows, got, want, data, n_samples, md, cell)
        # the oracle's paths on each slot's first row
        for n in ss.slots:
            k = next(k for k, (m, _) in enumerate(plan) if m == n)
            E = Expected(data[k], cell, block)
            assert E.root == rows[k][0].root, n
            for i, p, leaf in zip(got[0][k], got[1][k], got[2][k]):
                assert (p, leaf) == E.path(i, md), (n, i)
        # without cells the rest is the same
        assert ctx.prove_from_sources(rows, n_samples, md, cells=False) == got[:3] + ([[None] * n_samples] * len(rows),)
    finally:
        ss.free()


# ---- the one-slot case ------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("cell,block", [(64, 64), (2048, 65536), (100, 25600)], ids=["cpb1", "cpb32", "cpb256"])
def test_rows_of_one_slot_are_the_one_slot_call(pkg, ctx, torch_mod, tmp_path, cell, block):
    ss = SlotSet(pkg, ctx, torch_mod, tmp_path, cell, block)
    ss.fake("fake", 31 * cell + block, 8)
    ss.host("host", 37 * cell + block, 8)
    try:
        ent = [5, 6, 5, R - 2, 99]
        for slot, desc, _ in ss.slots.values():
            slot.compact()
            md = sum(slot.shape[2:]) + 1
            before = ctx.launches
            one = slot.prove_from_source(desc, ent, 16, md)
            mid = ctx.launches
            many = ctx.prove_from_sources([(slot, desc, e) for e in ent], 16, md)
            assert many == one
            assert ctx.launches - mid == mid - before
    finally:
        ss.free()


# ---- hundreds of slots: the launch count does not depend on their number -----------------------------------------

def launches_many(got, rows, cpb, block, block_depth, tile_mib):
    """kernel launches of a call on generated bytes with cells: indices, per tile of each source class (generator, sponge,
    cell gather), the sampled block trees, the check and the path gather"""
    tile = max(1, (tile_mib << 20) // block)
    n_tiles = 0
    for kind in (0, 1):
        pairs = {(id(rows[k][0]), i // cpb) for k in range(len(rows)) if rows[k][1][0] == kind for i in got[0][k]}
        if pairs:
            n_tiles += -(-len(pairs) // min(tile, len(pairs)))
    return 1 + 3 * n_tiles + (1 if cpb == 1 else block_depth) + 2


@gpu
def test_hundreds_of_slots_across_tiles(pkg, torch_mod):
    """256 compact 2 MiB slots (fake data and synthetic bytes), one challenge x 100 samples each, 16 MiB tiles: every row
    equals its slot's own answer, and the call launches the kernels of one pass per source class, for 256 slots as for 64"""
    torch = torch_mod
    ctx16 = fresh_context(pkg, CODEX_COMMIT_TILE_MIB=16)
    cell, block, n_blocks, M = 2048, 65536, 32, 256
    n_bytes = n_blocks * block
    slots = []
    try:
        d = torch.empty(M // 2 * n_bytes, dtype=torch.uint8, device="cuda")
        for m in range(M):
            seed = 0xC0FFEE + 7 * m
            if m % 2 == 0:
                slots.append((ctx16.slot_commit_fake(seed, n_bytes // cell, cell, block), (pkg.capi.SRC_FAKE, seed, n_bytes)))
            else:
                ptr = d.data_ptr() + (m // 2) * n_bytes
                ctx16.fill_synthetic_dev(seed, 0, n_bytes, ptr)
                torch.cuda.synchronize()
                slots.append((ctx16.slot_commit_dev(ptr, n_bytes, cell, block), (pkg.capi.SRC_SYNTHETIC, seed, n_bytes)))
        torch.cuda.synchronize()
        _, _, bd, sd = slots[0][0].shape
        md = bd + sd
        ent = [(0x9e3779b97f4a7c15 * (m + 1)) % R for m in range(M)]
        want = []
        for (slot, desc), e in zip(slots, ent):
            w = slot.prove_batch([e], 100, md)
            slot.compact()
            one = slot.prove_from_source(desc, [e], 100, md)
            assert one[:3] == w
            want.append(one)
        for m_rows in (M, M // 4):
            rows = [(slot, desc, e) for (slot, desc), e in zip(slots[:m_rows], ent)]
            before = ctx16.launches
            got = ctx16.prove_from_sources(rows, 100, md)
            launched = ctx16.launches - before
            for k in range(m_rows):
                assert tuple(part[k] for part in got) == tuple(part[0] for part in want[k]), k
            assert launched == launches_many(got, rows, block // cell, block, bd, 16), m_rows
            assert launched < 3 * m_rows                       # a pass per slot would launch at least 3 kernels per slot
    finally:
        for slot, _ in slots:
            slot.free()
        ctx16.close()


# ---- bytes that do not match ------------------------------------------------------------------------------------

@gpu
def test_mismatch_names_the_first_slot_and_its_smallest_block(pkg, ctx):
    capi = pkg.capi
    cell, block, n_blocks = 2048, 65536, 16
    n_bytes = n_blocks * block
    good = [ctx.slot_commit_fake(100 + m, n_bytes // cell, cell, block) for m in range(6)]
    host = random_bytes(41, n_bytes)
    hslot = ctx.slot_commit_host(host, cell, block)
    fslot = ctx.slot_commit_fake(77, n_bytes // cell, cell, block)
    try:
        for s in good + [hslot, fslot]:
            s.compact()
        n_cells = n_bytes // cell
        eh, ef1, ef2 = 1111, 2222, 3333
        first_h = ctx.cell_indices(eh, hslot.root, n_cells, 8)[0] // 32
        bad = host.copy()
        bad[first_h * block + 77] ^= 0x01
        f_blocks = {i // 32 for e in (ef1, ef2) for i in ctx.cell_indices(e, fslot.root, n_cells, 8)}
        g = [(s, (capi.SRC_FAKE, 100 + m, n_bytes), 50 + m) for m, s in enumerate(good)]
        h_row = (hslot, (capi.SRC_HOST, bad, n_bytes), eh)
        f_rows = [(fslot, (capi.SRC_FAKE, 78, n_bytes), ef1), (fslot, (capi.SRC_FAKE, 78, n_bytes), ef2)]
        # the fake slot's first row (3) comes before the host slot's (5): its smallest sampled block over both rows
        rows = g[:3] + [f_rows[0]] + g[3:4] + [h_row] + g[4:] + [f_rows[1]]
        expect_error(pkg, capi.CDX_ERR_MISMATCH, lambda: ctx.prove_from_sources(rows, 8, 32),
                     f"challenge 3: bytes of block {min(f_blocks)} do not hash to the committed block hash")
        # the host slot first
        rows = g[:2] + [h_row] + g[2:] + f_rows
        expect_error(pkg, capi.CDX_ERR_MISMATCH, lambda: ctx.prove_from_sources(rows, 8, 32),
                     f"challenge 2: bytes of block {first_h} do not hash to the committed block hash")
        # without those rows the call succeeds
        got = ctx.prove_from_sources(g, 8, 32)
        assert [r[0] for r in got[0]] == [ctx.cell_indices(e, s.root, n_cells, 1)[0] for s, _, e in g]
    finally:
        for s in good + [hslot, fslot]:
            s.free()


# ---- arguments --------------------------------------------------------------------------------------------------

@gpu
def test_refused_arguments(pkg, ctx, tmp_path):
    capi = pkg.capi
    cell, block = 2048, 65536
    host = random_bytes(12, 16 * block)
    small = ctx.slot_commit_host(host[:2 * block], cell, block)               # slot depth 1
    deep = ctx.slot_commit_host(host, cell, block)                            # slot depth 4
    other_geo = ctx.slot_commit_host(host[:2 * block], 1024, block)
    three = ctx.slot_commit_host(host[:3 * block], cell, block)
    ctx2 = pkg.Context(0)
    foreign = ctx2.slot_commit_host(host[:2 * block], cell, block)
    rng = ctx.slot_commit_range_host(host[:2 * block], cell, block, 0, 4, 0)
    comm = ctx.comm_init(1, 0, None)
    sharded = ctx.slot_commit_sharded_host(comm, host, 16 * block, cell, block, 0, 16, 2)
    d_small, d_deep = (capi.SRC_HOST, host, 2 * block), (capi.SRC_HOST, host, 16 * block)
    try:
        small.compact()
        _, _, bd, sd = deep.shape
        ok = [(small, d_small, 1), (deep, d_deep, 2)]
        call = ctx.prove_from_sources
        expect_error(pkg, capi.CDX_ERR_ARG, lambda: call([ok[0], (foreign, d_small, 3)], 4, 32), "challenge 1:")
        expect_error(pkg, capi.CDX_ERR_SIZE, lambda: call([ok[0], (other_geo, (capi.SRC_HOST, host, 2 * block), 3)], 4, 32), "challenge 1:")
        expect_error(pkg, capi.CDX_ERR_ARG, lambda: call(ok + [(small, (capi.SRC_HOST, host[block:], 2 * block), 3)], 4, 32), "challenge 2:")
        expect_error(pkg, capi.CDX_ERR_ARG, lambda: call(ok + [(small, (capi.SRC_FAKE, 1, 2 * block), 3)], 4, 32))
        expect_error(pkg, capi.CDX_ERR_STATE, lambda: call(ok + [(rng, (capi.SRC_HOST, host, 4 * block), 3)], 4, 32), "challenge 2:")
        expect_error(pkg, capi.CDX_ERR_STATE, lambda: call([(sharded, d_deep, 3)] + ok, 4, 32), "challenge 0:")
        expect_error(pkg, capi.CDX_ERR_NOT_POW2, lambda: call(ok + [(three, (capi.SRC_HOST, host, 3 * block), 3)], 4, 32))
        expect_error(pkg, capi.CDX_ERR_SIZE, lambda: call([ok[0], (deep, (capi.SRC_HOST, host, 8 * block), 2)], 4, 32))
        # max_depth: one below the deepest path is refused although the shallow slot's path fits
        expect_error(pkg, capi.CDX_ERR_RANGE, lambda: call(ok, 4, bd + sd - 1), "challenge 1:")
        expect_error(pkg, capi.CDX_ERR_RANGE, lambda: call(ok, 4, 65))
        got = call(ok, 4, bd + sd)
        assert all(p[bd + 1:] == [0] * (sd - 1) for p in got[1][0])              # the shallow slot's path is zero-padded
        missing = str(tmp_path / "missing.dat")
        expect_error(pkg, capi.CDX_ERR_ARG, lambda: call([ok[0], (deep, (capi.SRC_FILE, missing, 16 * block), 3)], 4, 32), missing)
        # more than 2^20 (challenge, sample) pairs
        expect_error(pkg, capi.CDX_ERR_SIZE, lambda: call(ok, (1 << 19) + 1, bd + sd, cells=False))
        # null pointers and zero challenges, through the C entry point
        lib = ctx.lib
        arr, keep = capi.make_descs([d_small])
        handles = (C.c_void_p * 1)(small.h)
        ent = capi._addr(capi.f2b(5))
        idx = (C.c_uint64 * 4)(*[0xAAAA] * 4)
        paths = C.create_string_buffer(b"\x5a" * (32 * 4 * 32), 32 * 4 * 32)
        args = [handles, arr, ent, 1, 4, 32, C.addressof(idx), C.addressof(paths), None, None]
        assert lib.cdx_slots_prove_from_source(*args) == capi.CDX_OK
        for a in (0, 1, 2, 6, 7):
            bad = list(args)
            bad[a] = None
            assert lib.cdx_slots_prove_from_source(*bad) == capi.CDX_ERR_ARG, a
        idx = (C.c_uint64 * 4)(*[0xAAAA] * 4)
        paths = C.create_string_buffer(b"\x5a" * (32 * 4 * 32), 32 * 4 * 32)
        assert lib.cdx_slots_prove_from_source(handles, arr, ent, 0, 4, 32, C.addressof(idx), C.addressof(paths), None, None) == capi.CDX_OK
        assert lib.cdx_slots_prove_from_source(None, None, None, 0, 4, 32, None, None, None, None) == capi.CDX_OK
        assert list(idx) == [0xAAAA] * 4 and paths.raw == b"\x5a" * (32 * 4 * 32)
        assert call([], 4, 32) == ([], [], [], [])
        del keep
    finally:
        for s in (small, deep, other_geo, three, rng, sharded):
            s.free()
        comm.destroy()
        foreign.free()
        ctx2.close()


# ---- guard bands ------------------------------------------------------------------------------------------------

@gpu
def test_many_slots_suite_within_guard_bands():
    """every GPU test above again with CODEX_COMMIT_GUARD=1 (4 KiB bands around every device allocation of the library,
    checked when it is freed): no write outside an allocation"""
    env = dict(os.environ, CODEX_COMMIT_GUARD="1")
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-x", "-q", "-k", "not within_guard_bands",
                          "-p", "no:cacheprovider"], capture_output=True, text=True, env=env, timeout=1500, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "CODEX_COMMIT_GUARD" not in res.stderr
    assert re.search(r"\b\d+ passed", res.stdout), res.stdout[-2000:]
