"""Compact commitments: a slot that keeps only its slot tree (cdx_slot_compact) answers challenges from the slot's bytes
(cdx_slot_prove_from_source), re-hashing only the sampled blocks.

Every answer must be byte for byte what cdx_slot_prove_batch gave on the same slot before compaction, at cells-per-block
1, 2, 32 and 256, on the TMA and the plain-load cell sponge, from every source kind and after both kinds of image import;
the returned cells must be the source's bytes; paths must match the oracle and reconstruct the root in two stages.  Also:
duplicate samples, sampled blocks spread over many tiles, what a compact handle refuses, the memory it saves, bytes that
do not match the commitment, compact images, and all of it again under CODEX_COMMIT_GUARD=1."""
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
HEADER_BYTES = 56                       # SlotImageHeader: magic, five uint64, two uint32

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
        self.cell, self.cpb = cell, block // cell
        self.root, bh, ch = coracle.commit_slot(bytes(data), cell, block, want_cells=True)
        self.trees = [coracle.merkle_layers(ch[b * self.cpb:(b + 1) * self.cpb]) for b in range(len(bh))]
        self.slot = coracle.merkle_layers(bh)
        self.block_depth, self.slot_depth = len(self.trees[0]) - 1, len(self.slot) - 1
        self.depth = self.block_depth + self.slot_depth

    def path(self, i, max_depth):
        merged = pyoracle.merge_merkle_proofs(pyoracle.merkle_proof(self.trees[i // self.cpb], i % self.cpb),
                                              pyoracle.merkle_proof(self.slot, i // self.cpb))
        return pyoracle.pad_merkle_proof(merged, max_depth).merkle_path, merged.leaf_value


def two_stage_roots(ctx, slot, idx, paths, leaves):
    """the verifier's view (Slot.hs:189-217): block trees from the leaves, then the slot tree from the block hashes"""
    n_cells, n_blocks, bd, sd = slot.shape
    cpb = n_cells // n_blocks
    flat_i = [i for ch in idx for i in ch]
    flat_p = [p for ch in paths for p in ch]
    flat_l = [v for ch in leaves for v in ch]
    blk = ctx.reconstruct_roots(flat_l, [i % cpb for i in flat_i], cpb, flat_p, bd)
    return ctx.reconstruct_roots(blk, [i // cpb for i in flat_i], n_blocks, [p[bd:] for p in flat_p], sd)


def check_compact_answers(pkg, ctx, slot, desc, data, E, entropies, n_samples=12):
    """prove_batch on the full slot, compact, prove_from_source: identical indices, paths, leaves; cells = source bytes;
    oracle paths on the first challenge; every answer reconstructs the root.  -> the full image taken before compaction"""
    n_cells, _, bd, sd = slot.shape
    cell = len(data) // n_cells
    md = bd + sd + 2
    want = slot.prove_batch(entropies, n_samples, md)
    image = slot.export()
    slot.compact()
    idx, paths, leaves, cells = slot.prove_from_source(desc, entropies, n_samples, md)
    assert (idx, paths, leaves) == want
    for k in range(len(entropies)):
        for i, c in zip(idx[k], cells[k]):
            assert c == bytes(data[i * cell:(i + 1) * cell]), (k, i)
    for i, p, leaf in zip(idx[0], paths[0], leaves[0]):
        assert (p, leaf) == E.path(i, md), i
    assert two_stage_roots(ctx, slot, idx, paths, leaves) == [E.root] * (len(entropies) * n_samples)
    # without cells the rest is the same
    assert slot.prove_from_source(desc, entropies[:1], n_samples, md, cells=False) == (idx[:1], paths[:1], leaves[:1], [[None] * n_samples])
    return image


# ---- equality with the full slot, every entry point ------------------------------------------------------------

@gpu
@pytest.mark.parametrize("cell,block", GEOMETRIES, ids=GEOMETRY_IDS)
def test_compact_answers_equal_full_slot(pkg, ctx, torch_mod, tmp_path, cell, block):
    torch = torch_mod
    capi = pkg.capi
    n_blocks = 8
    n_bytes, n_cells = n_blocks * block, n_blocks * block // cell
    entropies = [0, 1, R - 1, random.Random(cell * block).getrandbits(254) % R]
    seed = 1000003 * cell + block
    # the reference's fake data
    fake = ctx.fake_cells(seed, 0, n_cells, cell)
    E_fake = Expected(fake, cell, block)
    with ctx.slot_commit_fake(seed, n_cells, cell, block) as slot:
        full_image = check_compact_answers(pkg, ctx, slot, (capi.SRC_FAKE, seed, n_bytes), fake, E_fake, entropies)
        compact_image = slot.export()
    assert full_image[:8] == b"CDXSLOT1" and compact_image[:8] == b"CDXSLOTC"
    # both kinds of image
    with ctx.slot_import(full_image) as slot:
        assert check_compact_answers(pkg, ctx, slot, (capi.SRC_FAKE, seed, n_bytes), fake, E_fake, entropies) == full_image
    with ctx.slot_import(compact_image) as slot:
        idx, paths, leaves, cells = slot.prove_from_source((capi.SRC_FAKE, seed, n_bytes), entropies, 12, E_fake.depth + 2)
        for i, p, leaf, c in zip(idx[0], paths[0], leaves[0], cells[0]):
            assert (p, leaf) == E_fake.path(i, E_fake.depth + 2) and c == fake[i * cell:(i + 1) * cell]
        assert two_stage_roots(ctx, slot, idx, paths, leaves) == [E_fake.root] * (12 * len(entropies))
    # synthetic bytes on the device (cells at offsets that are not multiples of 8 where the geometry has them)
    syn = synthetic_ref(seed, n_bytes)
    d = torch.empty(n_bytes, dtype=torch.uint8, device="cuda")
    ctx.fill_synthetic_dev(seed, 0, n_bytes, d.data_ptr())
    torch.cuda.synchronize()
    with ctx.slot_commit_dev(d.data_ptr(), n_bytes, cell, block) as slot:
        check_compact_answers(pkg, ctx, slot, (capi.SRC_SYNTHETIC, seed, n_bytes), syn, Expected(syn, cell, block), entropies)
    # host memory and a file
    host = random_bytes(seed, n_bytes)
    E_host = Expected(host.tobytes(), cell, block)
    with ctx.slot_commit_host(host, cell, block) as slot:
        check_compact_answers(pkg, ctx, slot, (capi.SRC_HOST, host, n_bytes), host.tobytes(), E_host, entropies)
    path = str(tmp_path / "slot.dat")
    host.tofile(path)
    with ctx.slot_commit_file(path, n_bytes, 0, cell, block) as slot:
        check_compact_answers(pkg, ctx, slot, (capi.SRC_FILE, path, n_bytes), host.tobytes(), E_host, entropies)


@gpu
@pytest.mark.parametrize("cpb", [1, 2, 4])
def test_four_cell_slot_duplicate_samples(pkg, ctx, cpb):
    """4 cells, 64 samples: duplicate cells and blocks are certain; each block is hashed once and every sample still gets
    its own path and cell"""
    capi = pkg.capi
    cell = 64
    host = random_bytes(cpb, 4 * cell)
    E = Expected(host.tobytes(), cell, cell * cpb)
    with ctx.slot_commit_host(host, cell, cell * cpb) as slot:
        check_compact_answers(pkg, ctx, slot, (capi.SRC_HOST, host, 4 * cell), host.tobytes(), E, [7, 8, 9], n_samples=64)
    fake = ctx.fake_cells(99, 0, 4, cell)
    with ctx.slot_commit_fake(99, 4, cell, cell * cpb) as slot:
        check_compact_answers(pkg, ctx, slot, (capi.SRC_FAKE, 99, 4 * cell), fake, Expected(fake, cell, cell * cpb), [7, 8, 9], n_samples=64)


def launches_from_source(idx, cpb, block, block_depth, tile_mib):
    """kernel launches of a prove_from_source call on generated bytes with cells: indices, per tile (generator, sponge, cell
    gather), the sampled block trees, the check and the path gather"""
    n_unique = len({i // cpb for ch in idx for i in ch})
    tile = max(1, (tile_mib << 20) // block)
    n_tiles = -(-n_unique // min(tile, n_unique))
    return 1 + 3 * n_tiles + (1 if cpb == 1 else block_depth) + 2


@gpu
def test_thousand_challenges_across_tiles(pkg, torch_mod, tmp_path):
    """1000 challenges x 100 samples on a 256 MiB slot with 16 MiB tiles: the 4096 blocks are all sampled, many times each,
    and reach the sponge in 16 tiles; every source kind equals prove_batch, cells equal the slot bytes, and the launch
    count is that of the unique blocks"""
    import numpy as np
    torch = torch_mod
    capi = pkg.capi
    ctx16 = fresh_context(pkg, CODEX_COMMIT_TILE_MIB=16)
    try:
        cell, block, n_bytes, seed = 2048, 65536, 256 << 20, 0x5EED
        d = torch.empty(n_bytes, dtype=torch.uint8, device="cuda")
        ctx16.fill_synthetic_dev(seed, 0, n_bytes, d.data_ptr())
        torch.cuda.synchronize()
        host = d.cpu().numpy()
        path = str(tmp_path / "slot.dat")
        host.tofile(path)
        entropies = [(0x9e3779b97f4a7c15 * (k + 1)) % R for k in range(1000)]
        with ctx16.slot_commit_dev(d.data_ptr(), n_bytes, cell, block) as slot:
            n_cells, n_blocks, bd, sd = slot.shape
            want = slot.prove_batch(entropies, 100, 32)
            slot.compact()
            rows = host.reshape(n_cells, cell)
            for desc in ((capi.SRC_SYNTHETIC, seed, n_bytes), (capi.SRC_HOST, host, n_bytes), (capi.SRC_FILE, path, n_bytes)):
                before = ctx16.launches
                idx, paths, leaves, cells = slot.prove_from_source(desc, entropies, 100, 32)
                if desc[0] == capi.SRC_SYNTHETIC:
                    assert ctx16.launches - before == launches_from_source(idx, n_cells // n_blocks, block, bd, 16)
                assert (idx, paths, leaves) == want, desc[0]
                flat = np.array([i for ch in idx for i in ch], dtype=np.int64)
                got = np.frombuffer(b"".join(c for ch in cells for c in ch), dtype=np.uint8).reshape(-1, cell)
                assert np.array_equal(got, rows[flat]), desc[0]
            assert len({i // 32 for ch in want[0] for i in ch}) == n_blocks
            assert two_stage_roots(ctx16, slot, *want) == [slot.root] * 100000
    finally:
        ctx16.close()


# ---- state and memory -------------------------------------------------------------------------------------------

@gpu
def test_compact_slot_state_and_memory(pkg, ctx):
    capi = pkg.capi
    cell, block, n_blocks = 2048, 65536, 64
    host = random_bytes(3, n_blocks * block)
    with ctx.slot_commit_host(host, cell, block) as slot:
        n_cells, _, bd, sd = slot.shape
        full = slot.device_bytes
        shape, root = slot.shape, slot.root
        levels = [slot.read_layer(1, lvl, 0, max(1, n_blocks >> lvl)) for lvl in range(sd + 1)]
        blocks = slot.read_layer(0, bd, 0, n_blocks)
        slot.compact()
        compact = slot.device_bytes
        assert compact * 16 <= full
        assert full == 32 * (n_cells * 2 - n_blocks + (2 * n_blocks - 1) - n_blocks)     # forest + slot levels 1..depth
        assert compact == 32 * (2 * n_blocks - 1)
        slot.compact()                                                                    # compacting twice is fine
        assert slot.device_bytes == compact
        assert (slot.shape, slot.root) == (shape, root)
        assert [slot.read_layer(1, lvl, 0, max(1, n_blocks >> lvl)) for lvl in range(sd + 1)] == levels
        assert slot.read_layer(0, bd, 0, n_blocks) == blocks
        for call in (lambda: slot.cell_paths([0, 5], 32), lambda: slot.prove_batch([1], 4, 32), lambda: slot.read_layer(0, 0, 0, 1),
                     lambda: slot.read_layer(0, bd - 1, 0, 1)):
            with pytest.raises(pkg.CodexCommitError) as e:
                call()
            assert e.value.status == capi.CDX_ERR_STATE
        assert "prove_from_source" in ctx.lib.cdx_last_error(ctx.h).decode()
    # a range slot and a slot sharded above level 0 cannot be compacted or proven from their bytes
    with ctx.slot_commit_range_host(host, cell, block, 0, 2 * n_blocks, 0) as rng:
        for call in (rng.compact, lambda: rng.prove_from_source((capi.SRC_HOST, host, 2 * n_blocks * block), [1], 4, 32)):
            with pytest.raises(pkg.CodexCommitError) as e:
                call()
            assert e.value.status == capi.CDX_ERR_STATE
    comm = ctx.comm_init(1, 0, None)
    with ctx.slot_commit_sharded_host(comm, host, n_blocks * block, cell, block, 0, n_blocks, 2) as sh:
        with pytest.raises(pkg.CodexCommitError) as e:
            sh.compact()
        assert e.value.status == capi.CDX_ERR_STATE
    comm.destroy()
    # a dataset whose kept slot was compacted refuses to prove instead of reading released memory
    descs = [(capi.SRC_SYNTHETIC, 1, 2 * block), (capi.SRC_HOST, host, n_blocks * block)]
    with ctx.dataset_commit(None, descs, cell, block, keep_slot=1) as ds:
        ds.prove(5, 4, 32)
        assert ctx.lib.cdx_slot_compact(ctx.lib.cdx_dataset_kept_slot(ds.h)) == capi.CDX_OK
        with pytest.raises(pkg.CodexCommitError) as e:
            ds.prove(5, 4, 32)
        assert e.value.status == capi.CDX_ERR_STATE


# ---- bytes that do not match, and bad arguments -----------------------------------------------------------------

def expect_error(pkg, status, call, message=None):
    with pytest.raises(pkg.CodexCommitError) as e:
        call()
    assert e.value.status == status, str(e.value)
    if message:
        assert message in str(e.value), str(e.value)


@gpu
def test_mismatching_sources_and_bad_arguments(pkg, ctx, tmp_path):
    capi = pkg.capi
    cell, block, n_blocks = 2048, 65536, 16
    n_bytes = n_blocks * block
    host = random_bytes(11, n_bytes)
    path = str(tmp_path / "slot.dat")
    host.tofile(path)
    with ctx.slot_commit_host(host, cell, block) as slot:
        slot.compact()
        root, (n_cells, _, bd, sd) = slot.root, slot.shape
        entropy = [424242]
        sampled = sorted({i // 32 for i in ctx.cell_indices(entropy[0], root, n_cells, 8)})
        first = ctx.cell_indices(entropy[0], root, n_cells, 1)[0] // 32
        # one byte flipped inside the first sample's block
        bad = host.copy()
        bad[first * block + 1000] ^= 0x40
        expect_error(pkg, capi.CDX_ERR_MISMATCH, lambda: slot.prove_from_source((capi.SRC_HOST, bad, n_bytes), entropy, 8, 32),
                     f"bytes of block {first} do not hash")
        # a file cut at the start of the last sampled block: that block reads as zeros
        short = str(tmp_path / "short.dat")
        host[:sampled[-1] * block].tofile(short)
        expect_error(pkg, capi.CDX_ERR_MISMATCH, lambda: slot.prove_from_source((capi.SRC_FILE, short, n_bytes), entropy, 8, 32),
                     f"bytes of block {sampled[-1]} do not hash")
        # arguments
        expect_error(pkg, capi.CDX_ERR_SIZE, lambda: slot.prove_from_source((capi.SRC_HOST, host, n_bytes - block), entropy, 8, 32))
        expect_error(pkg, capi.CDX_ERR_ARG, lambda: slot.prove_from_source((capi.SRC_FILE, str(tmp_path / "missing.dat"), n_bytes), entropy, 8, 32))
        expect_error(pkg, capi.CDX_ERR_RANGE, lambda: slot.prove_from_source((capi.SRC_FILE, path, n_bytes), entropy, 8, bd + sd - 1))
        assert slot.prove_from_source((capi.SRC_FILE, path, n_bytes), entropy, 8, bd + sd)[0][0] == ctx.cell_indices(entropy[0], root, n_cells, 8)
    # the wrong fake seed: every sampled block differs, the smallest is named
    with ctx.slot_commit_fake(5, 16 * 32, cell, block) as slot:
        slot.compact()
        sampled = sorted({i // 32 for i in ctx.cell_indices(77, slot.root, 16 * 32, 8)})
        expect_error(pkg, capi.CDX_ERR_MISMATCH, lambda: slot.prove_from_source((capi.SRC_FAKE, 6, n_bytes), [77], 8, 32),
                     f"bytes of block {sampled[0]} do not hash")
        slot.prove_from_source((capi.SRC_FAKE, 5, n_bytes), [77], 8, 32)
    # three blocks: not a power-of-two cell count
    with ctx.slot_commit_host(host[:3 * block], cell, block) as slot:
        slot.compact()
        expect_error(pkg, capi.CDX_ERR_NOT_POW2, lambda: slot.prove_from_source((capi.SRC_HOST, host, 3 * block), [1], 4, 32))


# ---- images -----------------------------------------------------------------------------------------------------

@gpu
def test_compact_images(pkg, ctx):
    capi = pkg.capi
    cell, block, n_blocks = 256, 2048, 13                       # an odd block count: ragged slot levels
    host = random_bytes(21, n_blocks * block)
    with ctx.slot_commit_host(host, cell, block) as slot:
        n_cells, _, bd, sd = slot.shape
        forest = [v for lvl in range(bd + 1) for v in slot.read_layer(0, lvl, 0, n_cells >> lvl)]
        levels = [slot.read_layer(1, lvl, 0, -(-n_blocks // (1 << lvl))) for lvl in range(sd + 1)]
        full = slot.export()
        # the full image is what it always was: header, the whole forest, slot levels 1..depth
        assert full[:8] == b"CDXSLOT1" and full[HEADER_BYTES:] == capi.pack(forest + [v for lv in levels[1:] for v in lv])
        slot.compact()
        image = slot.export()
        assert len(image) == ctx.lib.cdx_slot_export_size(slot.h) == HEADER_BYTES + 32 * sum(len(lv) for lv in levels)
        assert image[:8] == b"CDXSLOTC" and image[HEADER_BYTES:] == capi.pack([v for lv in levels for v in lv])
        assert image[8:HEADER_BYTES - 24] == full[8:HEADER_BYTES - 24]       # cell, block size and block count
        assert int.from_bytes(image[32:40], "little") == 0                    # forest_nodes
    with ctx.slot_import(image) as back:
        assert back.export() == image
        assert back.device_bytes == 32 * sum(len(lv) for lv in levels)
        with pytest.raises(pkg.CodexCommitError) as e:
            back.prove_batch([1], 2, 16)
        assert e.value.status == capi.CDX_ERR_STATE
    with ctx.slot_import(full) as back:
        assert back.export() == full
    for broken, status in ((image[:-32], capi.CDX_ERR_SIZE), (image + b"\0" * 32, capi.CDX_ERR_SIZE), (b"CDXSLOTX" + image[8:], capi.CDX_ERR_ARG),
                           (image[:32] + (5).to_bytes(8, "little") + image[40:], capi.CDX_ERR_ARG), (image[:20], capi.CDX_ERR_SIZE)):
        expect_error(pkg, status, lambda: ctx.slot_import(broken))


# ---- guard bands ------------------------------------------------------------------------------------------------

@gpu
def test_compact_suite_within_guard_bands():
    """every GPU test above again with CODEX_COMMIT_GUARD=1 (4 KiB bands around every device allocation of the library,
    checked when it is freed): no write outside an allocation"""
    env = dict(os.environ, CODEX_COMMIT_GUARD="1")
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-x", "-q", "-k", "not within_guard_bands",
                          "-p", "no:cacheprovider"], capture_output=True, text=True, env=env, timeout=1500, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "CODEX_COMMIT_GUARD" not in res.stderr
    assert re.search(r"\b\d+ passed", res.stdout), res.stdout[-2000:]
