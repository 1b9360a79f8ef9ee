"""Retained tree levels and proof paths at every block geometry, against the oracle.

A slot commitment keeps three things besides its root: the block forest (cell hashes and every level of each block's
tree), the slot tree over the block hashes, and the cell paths gathered from both.  At the default geometry (2048-byte
cells, 32 cells per block) other tests check them closely; a bug that only changes a path, or a forest level above the
cell hashes, at another cells-per-block count (cpb) leaves every root intact.  This file compares all of them with the
oracle at cpb = 1 ... 256, through every entry point that builds or restores a slot.  It also covers the cell sponge
over every cell size the TMA loader takes up to 4 KiB and at every CTA width, the 64-bit index arithmetic of sampling
and root reconstruction, and the rule that element inputs >= r are taken mod r.

Part 0 (`expected_slot` and its CPU tests) needs no GPU: it checks the reference itself against pyoracle's proof-input
generator, so that the GPU tests below compare with something trustworthy."""
import concurrent.futures as cf
import functools
import importlib
import os
import random
import subprocess

import pytest

from conftest import PKG, ROOT
from oracle import coracle, pyoracle

gpu = pytest.mark.gpu
R = 21888242871839275222246405745257275088548364400416034343698204186575808495617
NONCANONICAL = (R, R + 1, 2**256 - 1)

# (cell bytes, block bytes): one-cell blocks (64/64, 2048/2048, 64 KiB/64 KiB), two-cell blocks (1024/2048, and 100/200
# on the plain-load kernel), 4 cells (2052/8208, plain loads), 8, 16, the default 32 as the control, 64, 128 (32/4096:
# cells below 64 bytes take the plain-load kernel) and 256 cells of 4 KiB per 1 MiB block (block_depth 8)
GEOMETRIES = [(64, 64), (2048, 2048), (65536, 65536), (1024, 2048), (100, 200), (2052, 8208), (256, 2048), (128, 2048),
              (2048, 65536), (64, 4096), (32, 4096), (4096, 1 << 20)]
GEOMETRY_IDS = [f"{c}x{b}" for c, b in GEOMETRIES]
N_BLOCKS = (1, 2, 3, 5, 8)


@pytest.fixture(scope="module", autouse=True)
def c_primitives(orc):
    """pyoracle's tree and proof code over the C oracle's hash primitives (same values, much faster)"""
    pyoracle.use_c_primitives(True)
    yield
    pyoracle.use_c_primitives(False)


# ---- 0. the expected values -------------------------------------------------------------------------------------

class ExpectedSlot:
    """What a committed slot of geometry (cell, block) must hold: cell hashes, every block-forest level, every
    slot-tree level, and the merged, padded path of any cell (gen_input/bn254.nim:53-74)."""

    def __init__(self, cell, block, cell_hashes, block_hashes, root):
        self.cell, self.block, self.cpb = cell, block, block // cell
        self.n_cells, self.n_blocks, self.root = len(cell_hashes), len(block_hashes), root
        cpb = self.cpb
        self.block_trees = [coracle.merkle_layers(cell_hashes[b * cpb:(b + 1) * cpb]) for b in range(self.n_blocks)]
        self.block_depth = len(self.block_trees[0]) - 1           # log2(cpb); 1 for one-cell blocks (the key-3 level)
        self.forest = [[v for t in self.block_trees for v in t[lvl]] for lvl in range(self.block_depth + 1)]
        assert self.forest[0] == cell_hashes and self.forest[-1] == block_hashes
        self.slot = coracle.merkle_layers(block_hashes)
        assert self.slot[-1] == [root]
        self.slot_depth = len(self.slot) - 1
        self.depth = self.block_depth + self.slot_depth
        self._paths = {}

    def path(self, i, max_depth):
        """(merkle path padded to max_depth, leaf) of cell i: merkleProof in the block tree and in the slot tree,
        merged, then padded with zeros (merkle.nim:21-42,86-100, types.nim:27-37)"""
        if i not in self._paths:
            cpb = self.cpb
            bot = pyoracle.merkle_proof(self.block_trees[i // cpb], i % cpb)
            top = pyoracle.merkle_proof(self.slot, i // cpb)
            merged = pyoracle.merge_merkle_proofs(bot, top)
            assert merged.leaf_index == i and merged.number_of_leaves == self.n_cells
            self._paths[i] = merged
        return pyoracle.pad_merkle_proof(self._paths[i], max_depth).merkle_path, self._paths[i].leaf_value

    def cells(self, limit, seed=0):
        """every cell when there are at most `limit`, otherwise the first and last cell of every block plus a seeded
        sample"""
        if self.n_cells <= limit:
            return list(range(self.n_cells))
        rnd = random.Random(seed)
        edges = {c for b in range(self.n_blocks) for c in (b * self.cpb, (b + 1) * self.cpb - 1)}
        return sorted(edges | set(rnd.sample(range(self.n_cells), min(limit, self.n_cells))))


def expected_slot(cell, block, data=None, seed=None, n_cells=None):
    """ExpectedSlot of the given slot bytes, or of the reference's fake data (slot.nim:23-32) for `seed`"""
    threads = min(8, os.cpu_count() or 1)
    if data is not None:
        root, bh, ch = coracle.commit_slot(data, cell, block, n_threads=threads, want_cells=True)
    else:
        root, bh, ch = coracle.commit_fake_slot(seed, n_cells, cell, block, n_threads=threads, want_cells=True)
    return ExpectedSlot(cell, block, ch, bh, root)


def fake_seed(cell, block, n_blocks):
    return 1000003 * cell + 7919 * block + n_blocks


@functools.lru_cache(maxsize=None)
def fake_expected(cell, block, n_blocks):
    """the slot every GPU test of this file commits at (cell, block, n_blocks), computed once"""
    return expected_slot(cell, block, seed=fake_seed(cell, block, n_blocks), n_cells=n_blocks * (block // cell))


def two_stage_root(E, i, path, leaf):
    """the verifier's view (Slot.hs:189-217): the block tree from the leaf, then the slot tree from the block hash"""
    blk = coracle.reconstruct_root(leaf, i % E.cpb, E.cpb, path[:E.block_depth])
    return blk, coracle.reconstruct_root(blk, i // E.cpb, E.n_blocks, path[E.block_depth:E.depth])


@pytest.mark.parametrize("cpb", [1, 2, 8, 64])
def test_expected_slot_agrees_with_generate_proof_input(cpb):
    """the helper against the reference's own proof-input generator (gen_input/bn254.nim:35-74) on the fake data:
    every block tree, the slot tree, and the merged padded path and leaf of every sampled cell"""
    cell, n_slots, slot_idx, entropy = 64, 3, 1, 0xC0FFEE
    n_cells = max(8, 4 * cpb)
    glob = pyoracle.GlobalConfig(max_depth=16, max_log2_nslots=2, cell_size=cell, block_size=cell * cpb)
    dset = pyoracle.DataSetConfig(n_slots=n_slots, n_cells=n_cells, n_samples=12, seed=4242)
    inp = pyoracle.generate_proof_input(glob, dset, slot_idx, entropy)
    seed = pyoracle.parametric_slot_seed(dset.seed, slot_idx)
    E = expected_slot(cell, cell * cpb, seed=seed, n_cells=n_cells)
    assert E.root == inp.slot_root
    assert E.block_depth == (1 if cpb == 1 else cpb.bit_length() - 1)
    mini, big = pyoracle.build_slot_tree_full(glob, n_cells, seed)
    assert E.block_trees == mini and E.slot == big
    idx = pyoracle.cell_indices(entropy, E.root, n_cells, dset.n_samples)
    for ci, proof, data in zip(idx, inp.merkle_proofs, inp.cell_data):
        assert E.path(ci, glob.max_depth) == (proof.merkle_path, proof.leaf_value)
        assert coracle.hash_bytes(data) == proof.leaf_value == E.forest[0][ci]
    # the same slot from its bytes instead of the seed
    data = b"".join(coracle.gen_fake_cell(seed, i, cell) for i in range(n_cells))
    B = expected_slot(cell, cell * cpb, data=data)
    assert (B.forest, B.slot) == (E.forest, E.slot)


@pytest.mark.parametrize("cpb", [1, 2, 8, 64])
@pytest.mark.parametrize("n_blocks", [1, 3, 5])
def test_expected_paths_reconstruct_in_two_stages(cpb, n_blocks):
    """every path of the helper, at ragged block counts too, walks back to its block hash and to the root, and is
    zero past the tree depth"""
    E = expected_slot(64, 64 * cpb, seed=cpb * 100 + n_blocks, n_cells=cpb * n_blocks)
    assert E.slot_depth == max(1, (n_blocks - 1).bit_length())
    for i in range(E.n_cells):
        path, leaf = E.path(i, E.depth + 2)
        assert leaf == E.forest[0][i]
        blk, root = two_stage_root(E, i, path, leaf)
        assert blk == E.slot[0][i // E.cpb] and root == E.root
        assert path[E.depth:] == [0, 0]


# ---- GPU helpers ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def plain_ctx(pkg):
    """a context whose cell sponge always takes the plain-load kernel (CODEX_COMMIT_PLAIN_LOADS=1)"""
    os.environ["CODEX_COMMIT_PLAIN_LOADS"] = "1"
    try:
        c = pkg.Context(0)
    finally:
        del os.environ["CODEX_COMMIT_PLAIN_LOADS"]
    yield c
    c.close()


def fake_dev(ctx, torch, E):
    d = torch.empty(E.n_cells * E.cell, dtype=torch.uint8, device="cuda")
    ctx.fake_cells_dev(fake_seed(E.cell, E.block, E.n_blocks), 0, E.n_cells, E.cell, d.data_ptr())
    torch.cuda.synchronize()
    return d


def check_layers(slot, E):
    """shape, every forest level 0..block_depth, every slot-tree level 0..slot_depth, root"""
    assert slot.shape == (E.n_cells, E.n_blocks, E.block_depth, E.slot_depth)
    for lvl, nodes in enumerate(E.forest):
        assert slot.read_layer(0, lvl, 0, len(nodes)) == nodes, ("forest", lvl)
    for lvl, nodes in enumerate(E.slot):
        assert slot.read_layer(1, lvl, 0, len(nodes)) == nodes, ("slot", lvl)
    assert slot.root == E.root


def check_paths(pkg, slot, E, cells, paths_fn=None):
    """paths and leaves at max_depth = the path length and 3 more (zero padding); one less is CDX_ERR_RANGE"""
    paths_fn = paths_fn or slot.cell_paths
    for max_depth in (E.depth, E.depth + 3):
        paths, leaves = paths_fn(cells, max_depth)
        for i, p, leaf in zip(cells, paths, leaves):
            assert (p, leaf) == E.path(i, max_depth), (i, max_depth)
    with pytest.raises(pkg.CodexCommitError) as e:
        paths_fn(cells[:1], E.depth - 1)
    assert e.value.status == pkg.capi.CDX_ERR_RANGE


def check_prove_batch(slot, E, entropies, n_samples=6):
    if E.n_cells & (E.n_cells - 1):
        return
    idx, paths, leaves = slot.prove_batch(entropies, n_samples, E.depth + 3)
    for k, e in enumerate(entropies):
        assert idx[k] == [coracle.cell_index(e % R, E.root, E.n_cells, c) for c in range(1, n_samples + 1)]
        for i, p, leaf in zip(idx[k], paths[k], leaves[k]):
            assert (p, leaf) == E.path(i, E.depth + 3)


# ---- 1. resident slots ------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("cell,block", GEOMETRIES, ids=GEOMETRY_IDS)
def test_resident_slot_layers_and_paths(ctx, pkg, torch_mod, cell, block):
    """slot_commit_fake and slot_commit_dev at n_blocks in {1, 2, 3, 5, 8}: every retained level, the path and leaf of
    every cell (a seeded sample with every block's first and last cell above 2048 cells), prove_batch"""
    torch = torch_mod
    for n_blocks in N_BLOCKS:
        E = fake_expected(cell, block, n_blocks)
        d = fake_dev(ctx, torch, E)
        cells = E.cells(2048, seed=n_blocks)
        entropies = [0, 1, 1234567, R - 1, random.Random(n_blocks).getrandbits(254) % R]
        for commit in (lambda: ctx.slot_commit_fake(fake_seed(cell, block, n_blocks), E.n_cells, cell, block),
                       lambda: ctx.slot_commit_dev(d.data_ptr(), E.n_cells * cell, cell, block)):
            with commit() as slot:
                check_layers(slot, E)
                check_paths(pkg, slot, E, cells)
                check_prove_batch(slot, E, entropies)


# ---- 2. the other entry points ----------------------------------------------------------------------------------

def ranges_at(n_blocks, world, top_level):
    """plan_block_ranges' split at a given exchange level: the 2^T-block chunks dealt out evenly, empty ranks included"""
    n_chunks = -(-n_blocks // (1 << top_level))
    out = []
    for r in range(world):
        b0 = min((n_chunks * r // world) << top_level, n_blocks)
        b1 = min((n_chunks * (r + 1) // world) << top_level, n_blocks)
        out.append((b0, b1 - b0))
    return out


def install_top(torch, shards):
    """single-GPU stand-in for the exchange inside cdx_slot_exchange_top: concatenate the level-T nodes of the emulated
    ranks and install them on each"""
    parts = []
    for s in shards:
        _, cnt, _ = s.subtree_roots()
        t = torch.empty(cnt * 32, dtype=torch.uint8, device="cuda")
        if cnt:
            s.subtree_roots_copy_dev(t.data_ptr())
        parts.append(t)
    torch.cuda.synchronize()
    gathered = torch.cat(parts).contiguous()
    for s in shards:
        s.set_top_dev(gathered.data_ptr(), gathered.numel() // 32)
    torch.cuda.synchronize()
    return gathered


def commit_in_ranges(ctx, torch, sharded, d, cell, block, n_blocks, ranges, top_level):
    """what the ranks do, back to back on one GPU: per-range commit, exchange of the level-T nodes, replicated top.
    Each range is copied to a buffer of its own (the device entry points want a 16-byte aligned base).  Ranks without
    blocks are skipped.  -> [(first, count, slot)]"""
    parts = [(first, count, d[first * block:(first + count) * block].clone()) for first, count in ranges if count]
    torch.cuda.synchronize()
    shards = [(first, count, ctx.slot_commit_range_dev(p.data_ptr(), count * block, cell, block, first, n_blocks, top_level))
              for first, count, p in parts]
    gathered = install_top(torch, [s for _, _, s in shards])
    assert gathered.numel() == 32 * sharded.level_width(n_blocks, top_level)
    return shards


def check_range_layers(slot, E, first, count, top_level):
    """a range's local forest and slot levels below T, and the global levels from T up"""
    for lvl, nodes in enumerate(E.forest):
        per_block = 1 if E.cpb == 1 else E.cpb >> lvl
        lo, n = first * per_block, count * per_block
        assert slot.read_layer(0, lvl, lo, n) == nodes[lo:lo + n], ("forest", lvl, first, count)
    for lvl, nodes in enumerate(E.slot):
        if lvl < top_level:
            lo, n = first >> lvl, -(-count // (1 << lvl))
            assert slot.read_layer(1, lvl, lo, n) == nodes[lo:lo + n], ("low", lvl, first, count)
        else:
            assert slot.read_layer(1, lvl, 0, len(nodes)) == nodes, ("top", lvl, first, count)
    assert slot.root == E.root


@gpu
@pytest.mark.parametrize("cell,block", GEOMETRIES, ids=GEOMETRY_IDS)
def test_other_entry_points_layers_and_paths(ctx, pkg, torch_mod, tmp_path, cell, block):
    """the same slots through slot_commit_host (pageable and pinned), slot_commit_file, export/slot_import, the sharded
    protocol emulated on one GPU (ranges of plan_block_ranges for 2, 3 and 8 ranks, at T = 0, 1, slot_depth and the
    planned T), slot_commit_sharded_dev on a one-rank communicator, and dataset_commit with the slot kept: the same
    levels and paths as the oracle"""
    torch = torch_mod
    capi = pkg.capi
    sharded = importlib.import_module(PKG + ".sharded")
    comm = ctx.comm_init(1, 0, None)
    for n_blocks in N_BLOCKS:
        E = fake_expected(cell, block, n_blocks)
        n_bytes = E.n_cells * cell
        d = fake_dev(ctx, torch, E)
        host = d.cpu().numpy()
        cells = E.cells(64, seed=n_blocks)
        pinned = torch.empty(n_bytes, dtype=torch.uint8, pin_memory=True)
        pinned.copy_(d)
        torch.cuda.synchronize()
        path = str(tmp_path / "slot.dat")
        host.tofile(path)
        commits = [lambda: ctx.slot_commit_host(host, cell, block),
                   lambda: ctx.slot_commit_host(pinned.data_ptr(), cell, block, n_bytes=n_bytes),
                   lambda: ctx.slot_commit_file(path, n_bytes, 0, cell, block)]
        for commit in commits:
            with commit() as slot:
                check_layers(slot, E)
                check_paths(pkg, slot, E, cells)
        with ctx.slot_commit_dev(d.data_ptr(), n_bytes, cell, block) as live:
            image = live.export()
        with ctx.slot_import(image) as back:
            check_layers(back, E)
            check_paths(pkg, back, E, cells)
            check_prove_batch(back, E, [5, R - 2])
        # the sharded protocol, one rank after the other
        levels = [0] if n_blocks == 1 else sorted({0, 1, E.slot_depth})
        for world in (2, 3, 8):
            planned_t, planned = sharded.plan_block_ranges(n_blocks, world)
            for top_level in sorted(set(levels) | {planned_t}):
                ranges = planned if top_level == planned_t else ranges_at(n_blocks, world, top_level)
                assert capi.block_ranges_top_level(n_blocks, ranges) >= top_level
                shards = commit_in_ranges(ctx, torch, sharded, d, cell, block, n_blocks, ranges, top_level)
                for first, count, s in shards:
                    check_range_layers(s, E, first, count, top_level)
                # the owner of a cell returns its whole path and leaf, every other range zeros: the sum is the path
                got = [s.cell_paths(cells, E.depth + 3) for _, _, s in shards]
                for k, i in enumerate(cells):
                    want = E.path(i, E.depth + 3)
                    for (first, count, _), (paths, leaves) in zip(shards, got):
                        mine = first * E.cpb <= i < (first + count) * E.cpb
                        assert (paths[k], leaves[k]) == (want if mine else ([0] * (E.depth + 3), 0)), (world, top_level, i)
                for _, _, s in shards:
                    s.free()
        for top_level in levels:
            with ctx.slot_commit_sharded_dev(comm, d.data_ptr(), n_bytes, cell, block, 0, n_blocks, top_level) as sh:
                check_layers(sh, E)
                check_paths(pkg, sh, E, cells, paths_fn=lambda c, m: sh.cell_paths_sharded(comm, c, m))
                check_paths(pkg, sh, E, cells)
        # a dataset that keeps this slot: ds.prove gives the oracle's indices, paths and leaves
        if E.n_cells & (E.n_cells - 1) == 0:
            descs = [(capi.SRC_SYNTHETIC, 11, 2 * block), (capi.SRC_HOST, host, n_bytes), (capi.SRC_SYNTHETIC, 12, 3 * block)]
            with ctx.dataset_commit(None, descs, cell, block, keep_slot=1) as ds:
                roots = ds.slot_roots
                assert roots[1] == E.root and ds.root == coracle.merkle_root(roots)
                for entropy in (77, R + 77):
                    idx, paths, leaves = ds.prove(entropy, 5, E.depth + 2)
                    assert idx == [coracle.cell_index(entropy % R, E.root, E.n_cells, c) for c in range(1, 6)]
                    for i, p, leaf in zip(idx, paths, leaves):
                        assert (p, leaf) == E.path(i, E.depth + 2), (entropy, i)
    comm.destroy()


# ---- 3. the cell sponge across cell sizes and CTA widths --------------------------------------------------------

def synthetic(ctx, torch, n_bytes, seed):
    d = torch.empty((n_bytes + 7) // 8 * 8, dtype=torch.uint8, device="cuda")
    ctx.fill_synthetic_dev(seed, 0, d.numel(), d.data_ptr())
    torch.cuda.synchronize()
    return d


def hash_cells(ctx, torch, d, n_cells, cell):
    out = torch.empty(32 * n_cells, dtype=torch.uint8, device="cuda")
    ctx.hash_cells_dev(d.data_ptr(), n_cells, cell, out.data_ptr())
    torch.cuda.synchronize()
    return out


def oracle_cell_hashes(host, cell, cells):
    threads = min(16, os.cpu_count() or 1)
    with cf.ThreadPoolExecutor(threads) as ex:                       # ctypes releases the GIL inside the oracle
        return list(ex.map(lambda i: coracle.hash_bytes(host[i * cell:(i + 1) * cell]), cells))


def unpack(out):
    return coracle.unpack(out.cpu().numpy().tobytes())


@gpu
def test_cell_sponge_every_tma_cell_size(ctx, torch_mod):
    """every multiple of 32 from 64 to 4096 bytes (the TMA loader's row ring: segment clamp at the last segment, the
    synthesized pad word) with a partial last warp, every cell against the oracle"""
    torch = torch_mod
    n_cells = 45
    d = synthetic(ctx, torch, n_cells * 4096, seed=32)
    host = d.cpu().numpy().tobytes()
    for cell in range(64, 4097, 32):
        got = unpack(hash_cells(ctx, torch, d, n_cells, cell))
        assert got == oracle_cell_hashes(host, cell, range(n_cells)), cell


@gpu
def test_cell_sponge_every_plain_cell_size(plain_ctx, torch_mod):
    """every multiple of 4 from 4 to 1024 bytes on the plain-load kernel, every cell against the oracle"""
    torch = torch_mod
    n_cells = 37
    d = synthetic(plain_ctx, torch, n_cells * 1024, seed=4)
    host = d.cpu().numpy().tobytes()
    for cell in range(4, 1025, 4):
        got = unpack(hash_cells(plain_ctx, torch, d, n_cells, cell))
        assert got == oracle_cell_hashes(host, cell, range(n_cells)), cell


@gpu
def test_cell_sponge_at_every_cta_width(ctx, plain_ctx, torch_mod):
    """cell counts at both ends of each CTA width the launch picks (256, 128, 64, 32 threads: narrower CTAs while a
    launch has fewer than sm_count CTAs' worth of cells), thresholds from the device's SM count: all cells equal the
    plain-load kernel's, a seeded sample equals the oracle"""
    torch = torch_mod
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    counts = [sm * 256, sm * 256 + 33, sm * 128, sm * 256 - 1, sm * 64, sm * 128 - 1, 33, sm * 64 - 1]
    for cell in (64, 160, 2048):
        d = synthetic(ctx, torch, max(counts) * cell, seed=cell)
        host = d.cpu().numpy().tobytes()
        for n_cells in counts:
            a, b = hash_cells(ctx, torch, d, n_cells, cell), hash_cells(plain_ctx, torch, d, n_cells, cell)
            assert torch.equal(a, b), (cell, n_cells)
            rnd = random.Random(n_cells)
            sample = sorted({0, n_cells - 1} | set(rnd.sample(range(n_cells), 30)))
            got = coracle.unpack(b"".join(a[32 * i:32 * i + 32].cpu().numpy().tobytes() for i in sample))
            assert got == oracle_cell_hashes(host, cell, sample), (cell, n_cells)


@gpu
def test_cell_sponge_large_cells(ctx, plain_ctx, torch_mod):
    """8 KiB, 64 KiB, 1 MiB - 32 and 1 MiB cells, 33 of each, on both loaders and against the oracle"""
    torch = torch_mod
    n_cells = 33
    for cell in (8192, 65536, (1 << 20) - 32, 1 << 20):
        d = synthetic(ctx, torch, n_cells * cell, seed=cell)
        host = d.cpu().numpy().tobytes()
        a, b = hash_cells(ctx, torch, d, n_cells, cell), hash_cells(plain_ctx, torch, d, n_cells, cell)
        assert torch.equal(a, b), cell
        assert unpack(a) == oracle_cell_hashes(host, cell, range(n_cells)), cell


# ---- 4. index widths and the mod-r contract ---------------------------------------------------------------------

@gpu
def test_cell_indices_at_every_index_width(ctx):
    """numberOfCells = 2^k up to 2^63: the index keeps the low k bits of the sponge output, high word included"""
    rnd = random.Random(64)
    for k in (0, 1, 31, 32, 33, 40, 63):
        for _ in range(3):
            entropy, root = rnd.randrange(R), rnd.randrange(R)
            got = ctx.cell_indices(entropy, root, 1 << k, 64)
            assert got == [coracle.cell_index(entropy, root, 1 << k, c) for c in range(1, 65)], k
            assert all(i < (1 << k) for i in got)
        if k >= 33:
            assert any(i >> 32 for i in got), k


@gpu
def test_noncanonical_entropies_and_roots(ctx, pkg):
    """entropy and slot root in {0, 1, r-1, r, r+1, 2^256-1} are taken mod r, in cell_indices and in prove_batch"""
    values = (0, 1, R - 1) + NONCANONICAL
    n = 1 << 40
    for e in values:
        for root in values:
            assert ctx.cell_indices(e, root, n, 8) == [coracle.cell_index(e % R, root % R, n, c) for c in range(1, 9)], (e, root)
    E = fake_expected(256, 2048, 8)
    with ctx.slot_commit_fake(fake_seed(256, 2048, 8), E.n_cells, 256, 2048) as slot:
        check_prove_batch(slot, E, list(values), n_samples=8)


@gpu
def test_reconstruct_roots_with_64_bit_leaf_counts(ctx):
    """trees of 2^32 + 1 ... 2^63 - 1 leaves (index and width walked as 64-bit values, odd nodes at high levels),
    path_stride > depth with nonzero junk past the depth, against reconstructRoot (merkle.nim:51-74)"""
    rnd = random.Random(63)
    for n in (2**32 + 1, 2**40 - 1, 2**62 + 3, 2**63 - 1):
        depth = (n - 1).bit_length()
        idx = [0, n - 1, n - 2, 2**32] + [rnd.randrange(n) for _ in range(12)]
        leaves = [rnd.randrange(R) for _ in idx]
        paths = [[rnd.randrange(R) for _ in range(depth)] + [rnd.randrange(1, R) for _ in range(3)] for _ in idx]
        got = ctx.reconstruct_roots(leaves, idx, n, paths, depth=depth)
        assert got == [coracle.reconstruct_root(lf, i, n, p[:depth]) for lf, i, p in zip(leaves, idx, paths)], n


@gpu
def test_noncanonical_elements_are_taken_mod_r(ctx):
    """sponge, keyed compression, Merkle layers and root, and root reconstruction (leaf and path) with elements r, r+1
    and 2^256-1 equal the oracle on the values mod r; every output is canonical"""
    rnd = random.Random(256)
    pool = list(NONCANONICAL) + [rnd.randrange(R) for _ in range(3)]
    for ln in (1, 2, 3, 4, 7):
        items = [[rnd.choice(pool) for _ in range(ln)] for _ in range(6)] + [[x] * ln for x in NONCANONICAL]
        for rate in (1, 2):
            assert ctx.sponge_batch(items, rate) == [coracle.sponge([x % R for x in it], rate) for it in items], (ln, rate)
    xs = [x for x in NONCANONICAL for _ in range(4)]
    ys = [y for _ in range(4) for y in NONCANONICAL]
    xs, ys = xs + xs[:4], ys + ys[:4]
    keys = [k % 4 for k in range(len(xs))]
    assert ctx.compress_batch(xs, ys, keys) == [coracle.compress(x % R, y % R, k) for x, y, k in zip(xs, ys, keys)]
    for n in (1, 2, 3, 5, 8):
        leaves = [rnd.choice(pool) for _ in range(n)]
        want = coracle.merkle_layers([x % R for x in leaves])
        assert ctx.merkle_layers(leaves) == want, n
        assert ctx.merkle_layers(leaves, bottom=False) == coracle.merkle_layers([x % R for x in leaves], False), n
        assert ctx.merkle_root(leaves) == want[-1][0], n
    n = 13
    idx = list(range(n))
    leaves = [rnd.choice(pool) for _ in idx]
    paths = [[rnd.choice(pool) for _ in range(4)] for _ in idx]
    assert ctx.reconstruct_roots(leaves, idx, n, paths) == \
        [coracle.reconstruct_root(lf % R, i, n, [p % R for p in ps]) for lf, i, ps in zip(leaves, idx, paths)]


# ---- 5. the cli at other geometries -----------------------------------------------------------------------------

def run_cli(args, tmp_path):
    cli = os.path.join(ROOT, "codex-storage-proofs-circuits_b200", "cli")
    assert os.path.exists(cli), "build the host cli first (__graft_entry__.build())"
    out = str(tmp_path / "input.json")
    res = subprocess.run([cli] + args + ["--output=" + out], capture_output=True, text=True)
    return res, out


@gpu
@pytest.mark.parametrize("cell,block,n_cells,n_slots,index", [(256, 2048, 128, 3, 2), (1024, 2048, 64, 5, 4),
                                                               (4096, 262144, 256, 2, 1), (512, 512, 64, 3, 0)])
def test_cli_other_geometries(tmp_path, cell, block, n_cells, n_slots, index):
    """cli -> input.json at other cell and block sizes: byte-identical to pyoracle's generator, accepted by --selfcheck,
    and accepted by the circuit restatement -- except with one-cell blocks (512/512).  There the Nim generator's
    one-leaf block tree has a key-3 level, so every merged path starts with one zero sibling (block_depth 1), while the
    circuit's main component takes blockTreeDepth = log2(cpb) = 0 (cli.nim:186-204, sample_cells.circom) and walks the
    slot tree from the bare cell hash: the circuit rejects what the reference's generator writes.  The library keeps
    the generator's path shape; this test pins both sides of that inconsistency."""
    from oracle import circuit_verifier as cv
    depth, max_slots, n_samples, seed, entropy = 20, 8, 6, 4321, 98765
    args = (f"--field=bn254 --hash=poseidon2 --cellsize={cell} --blocksize={block} --ncells={n_cells} --nslots={n_slots} "
            f"--index={index} --nsamples={n_samples} --seed={seed} --entropy={entropy} --depth={depth} --maxslots={max_slots} "
            "--selfcheck").split()
    res, out = run_cli(args, tmp_path)
    assert res.returncode == 0, res.stderr
    assert "selfcheck: the proof input satisfies every constraint" in res.stdout
    txt = open(out).read()
    glob = pyoracle.GlobalConfig(max_depth=depth, max_log2_nslots=pyoracle.ceiling_log2(max_slots), cell_size=cell, block_size=block)
    dset = pyoracle.DataSetConfig(n_slots=n_slots, n_cells=n_cells, n_samples=n_samples, seed=seed)
    assert txt == pyoracle.export_proof_input(pyoracle.generate_proof_input(glob, dset, index, entropy))
    if block == cell:
        with pytest.raises(AssertionError, match="middle/bottom root check failed"):
            cv.verify_input_json(txt, depth, 3, cell, block)
    else:
        cv.verify_input_json(txt, depth, 3, cell, block)
