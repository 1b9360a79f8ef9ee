"""Many slots in one call: the batched entry points (cdx_slots_commit_batch_*) and the dataset commitment
(cdx_dataset_commit) across batch boundaries, and synthetic slot bytes at any offset.

CPU: a Python restatement of how cdx_dataset_commit splits a rank's slots -- the LPT plan, the whole/batched rule
(<= 64 MiB and not the kept slot), the 1 GiB flush -- checked against cdx_dataset_plan, and of the kernel launches such a
commit makes.
GPU: thousands of slot trees in one segmented level pass (k_merkle_level_seg) against the oracle; a dataset of 1.1 GiB
whose first batch fills the 1 GiB cap exactly, whose batch roots are scattered back from LPT order into slot order, with
every source kind; synthetic members whose size or start is not a multiple of 8 (a batch member behind a 300-byte one, a
tile that starts inside a word)."""
import concurrent.futures as cf
import importlib
import os
import random

import pytest

from conftest import PKG

SMALL_BYTES, BATCH_CAP = 64 << 20, 1 << 30                # cdx_dataset_commit: batched slots, bytes per batch


@pytest.fixture(scope="module")
def capi(pkg):
    return pkg.capi


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


def synthetic_ref(seed, first, n):
    """bytes [first, first + n) of a synthetic slot: byte b is byte b % 8 of splitmix64(seed + b / 8), little-endian"""
    import bench
    return bench.synthetic_bytes_host(seed, 0, (first + n + 7) // 8 * 8)[first:first + n].copy()


def random_bytes(seed, n):
    import numpy as np
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8)


def oracle_roots(orc, parts, cell, block, workers=None):
    """orc.commit_slot over many small byte arrays, spread over threads (the oracle releases the GIL)"""
    with cf.ThreadPoolExecutor(workers or os.cpu_count() or 4) as ex:
        return list(ex.map(lambda p: orc.commit_slot((p.ctypes.data, p.nbytes), cell, block)[0], parts))


class BorrowedSlot:
    """read access to a slot the caller does not own (a dataset's kept slot): never freed through this handle"""

    def __init__(self, pkg, ctx, h):
        self.slot = pkg.capi.Slot(ctx, h)

    def __enter__(self):
        return self.slot

    def __exit__(self, *a):
        self.slot.h = None


def raw_layer(ctx, h, tree, level, first, count):
    import ctypes as C
    out = C.create_string_buffer(32 * count)
    ctx._chk(ctx.lib.cdx_slot_read_layer(h, tree, level, first, count, C.addressof(out)))
    return out.raw


# ---- the partition of a dataset commit, restated -----------------------------------------------------------------

def plan_dataset(blocks, n_ranks, block_size):
    """plan_dataset in capi_multi.cuh: LPT (largest first, stable by index, onto the least loaded rank, lowest rank on a
    tie); a slot of at least 256 MiB per rank that alone exceeds a quarter of a rank's share is sharded (owner -1)"""
    total = sum(blocks)
    min_shard = max(1, (256 << 20) // block_size) * n_ranks
    owner, mine, load = [0] * len(blocks), [[] for _ in range(n_ranks)], [0] * n_ranks
    for k in sorted(range(len(blocks)), key=lambda i: (-blocks[i], i)):
        if n_ranks > 1 and blocks[k] >= min_shard and blocks[k] * 4 * n_ranks > total:
            owner[k] = -1
            continue
        r = min(range(n_ranks), key=lambda j: (load[j], j))
        owner[k] = r
        mine[r].append(k)
        load[r] += blocks[k]
    return owner, mine


def partition(mine, slot_bytes, keep=-1):
    """one rank's own slots -> (whole slots, batches), in commit order: a slot goes to the open batch if it has at most
    64 MiB and is not the kept one; the batch is flushed first if the slot would take it past 1 GiB"""
    whole, batches, cur, cur_bytes = [], [], [], 0
    for k in mine:
        if k != keep and slot_bytes[k] <= SMALL_BYTES:
            if cur_bytes + slot_bytes[k] > BATCH_CAP:
                batches.append(cur)
                cur, cur_bytes = [], 0
            cur.append(k)
            cur_bytes += slot_bytes[k]
        else:
            whole.append(k)
    if cur:
        batches.append(cur)
    return whole, batches


def seg_launches(slot_blocks):
    """k_merkle_level_seg launches of batch_trees: one per level until every slot tree has its root (a one-block tree
    still gets its key-3 compression)"""
    w, level, levels = list(slot_blocks), 0, 0
    while sum(w):
        levels += 1
        w = [0 if level > 0 and x <= 1 else (x + 1) // 2 for x in w]
        level += 1
    return levels - 1


def tree_launches(n):
    """k_merkle_level launches of merkle_layers_on_device over n leaves with the bottom-layer rule"""
    launches, bottom = 0, True
    while bottom or n > 1:
        n, bottom = (n + 1) // 2, False
        launches += 1
    return launches


def batch_launches(slot_blocks, cpb):
    """one batch of host-memory members: the cell sponge, the block forest, the segmented slot levels, the root scatter"""
    forest = 1 if cpb == 1 else cpb.bit_length() - 1
    return 1 + forest + seg_launches(slot_blocks) + 1


def draw_mix(rnd, n_slots, block_size):
    """slot sizes in bytes around the thresholds: one-block slots, slots at and just above 64 MiB, huge slots that the
    sharding rule takes on several ranks"""
    per_64m = SMALL_BYTES // block_size
    picks = [lambda: 1, lambda: rnd.randint(2, 70), lambda: rnd.randint(71, per_64m - 1), lambda: per_64m, lambda: per_64m + 1,
             lambda: rnd.randint(per_64m + 2, 40 * per_64m), lambda: rnd.randint(1, 400) * (1 << 30) // block_size]
    return [block_size * rnd.choice(picks)() for _ in range(n_slots)]


@pytest.mark.parametrize("n_ranks", [1, 2, 3, 8])
def test_partition_restatement_matches_library_plan(capi, n_ranks):
    rnd = random.Random(1000 + n_ranks)
    for case in range(40):
        block = rnd.choice([65536, 2048, 100, 36 * 2])
        sizes = draw_mix(rnd, rnd.randint(1, 300), block)
        owner, mine = plan_dataset([s // block for s in sizes], n_ranks, block)
        assert capi.dataset_plan(sizes, n_ranks, block) == owner, (n_ranks, case)
        keep = rnd.randrange(-1, len(sizes))
        for r in range(n_ranks):
            assert mine[r] == sorted((k for k in range(len(sizes)) if owner[k] == r), key=lambda k: (-sizes[k], k))
            whole, batches = partition(mine[r], sizes, keep)
            assert sorted(whole + [k for b in batches for k in b]) == sorted(mine[r])
            for i, b in enumerate(batches):
                assert sum(sizes[k] for k in b) <= BATCH_CAP and all(sizes[k] <= SMALL_BYTES and k != keep for k in b)
                if i + 1 < len(batches):                                   # flushed only because the next slot did not fit
                    assert sum(sizes[k] for k in b) + sizes[batches[i + 1][0]] > BATCH_CAP
            assert all(sizes[k] > SMALL_BYTES or k == keep for k in whole)


def test_launch_restatement_small_cases():
    assert [seg_launches([b]) for b in (1, 2, 3, 4, 5, 64, 65, 1024, 1025)] == [1, 1, 2, 2, 3, 6, 7, 10, 11]
    assert seg_launches([1, 1024, 2, 64]) == 10 and seg_launches([1] * 5) == 1
    assert [tree_launches(n) for n in (1, 2, 3, 13, 256, 257)] == [1, 1, 2, 4, 8, 9]
    assert batch_launches([1, 3], 1) == 1 + 1 + 2 + 1 and batch_launches([64] * 3, 32) == 1 + 5 + 6 + 1


# ---- the big mix: 1.1 GiB, two batches, every source kind ----------------------------------------------------------

MIB4, BLOCK, CELL = 64, 65536, 2048                        # 4 MiB = 64 blocks of 64 KiB


def big_mix():
    """(kind, blocks, extra) per slot, in a shuffled index order (so that LPT order is not index order), and the index
    of the kept slot.  LPT puts the 64 MiB slot first among the batched ones: it and the 240 slots of 4 MiB fill the
    first batch to exactly 1 GiB; the 2 MiB slot opens the second batch, which holds nothing deeper than 32 blocks (so a
    batch flushed one slot early would launch one more segmented level)."""
    members = [("syn", MIB4, None)] * 240 + [("syn", 1024, None), ("syn", 1025, None), ("syn", 32, None), ("keep", 16, None),
                                              ("syn", 1, None), ("syn", 3, None), ("fake", 5, None), ("host", 7, None),
                                              ("host", 2, None), ("file", 9, None), ("file", 11, 6 * BLOCK + 1234), ("fake", 13, None)]
    rnd = random.Random(4242)
    rnd.shuffle(members)
    keep = [m[0] for m in members].index("keep")
    return members, keep


def test_big_mix_partition():
    members, keep = big_mix()
    sizes = [b * BLOCK for _, b, _ in members]
    owner, mine = plan_dataset([b for _, b, _ in members], 1, BLOCK)
    whole, batches = partition(mine[0], sizes, keep)
    assert sorted(sizes[k] for k in whole) == [16 * BLOCK, 1025 * BLOCK]
    assert [sum(sizes[k] for k in b) for b in batches] == [BATCH_CAP, (32 + 1 + 3 + 5 + 7 + 2 + 9 + 11 + 13) * BLOCK]
    assert sizes[batches[0][0]] == SMALL_BYTES and sizes[batches[1][0]] == 32 * BLOCK
    assert mine[0] != sorted(mine[0])                                        # LPT order is not index order


@pytest.mark.gpu
def test_dataset_across_batch_boundaries(pkg, capi, ctx, orc, torch_mod, tmp_path):
    torch = torch_mod
    import numpy as np
    members, keep = big_mix()
    n = len(members)
    sizes = [b * BLOCK for _, b, _ in members]
    whole, batches = partition(plan_dataset([b for _, b, _ in members], 1, BLOCK)[1][0], sizes, keep)
    descs, host_bytes = [], {}                                              # host_bytes: the bytes the oracle sees
    for k, (kind, b, extra) in enumerate(members):
        seed = 0x5000 + 7 * k
        if kind in ("syn", "keep"):
            descs.append((capi.SRC_SYNTHETIC, seed, sizes[k]))
        elif kind == "fake":
            descs.append((capi.SRC_FAKE, seed, sizes[k]))
        elif kind == "host":
            host_bytes[k] = random_bytes(seed, sizes[k])
            descs.append((capi.SRC_HOST, host_bytes[k], sizes[k]))
        else:
            data = random_bytes(seed, extra or sizes[k])
            path = str(tmp_path / f"slot{k}.dat")
            data.tofile(path)                                               # a short file reads as zeros past its end
            host_bytes[k] = np.concatenate([data, np.zeros(sizes[k] - data.size, np.uint8)])
            descs.append((capi.SRC_FILE, path, sizes[k]))
    with ctx.dataset_commit(None, descs, CELL, BLOCK, keep_slot=keep) as ds:
        roots = ds.slot_roots
        assert ds.stats == {"bytes_local": sum(sizes), "whole": len(whole), "batched": sum(len(b) for b in batches), "sharded": 0}
        # every slot root: the single-slot GPU commit of the same source
        for k, (kind, b, _) in enumerate(members):
            if descs[k][0] == capi.SRC_SYNTHETIC:
                d = torch.empty(sizes[k], dtype=torch.uint8, device="cuda")
                ctx.fill_synthetic_dev(descs[k][1], 0, sizes[k], d.data_ptr())
                with ctx.slot_commit_dev(d.data_ptr(), sizes[k]) as s:
                    assert roots[k] == s.root, k
            elif kind == "fake":
                with ctx.slot_commit_fake(descs[k][1], sizes[k] // CELL) as s:
                    assert roots[k] == s.root, k
            elif kind == "host":
                with ctx.slot_commit_host(host_bytes[k]) as s:
                    assert roots[k] == s.root, k
            else:
                with ctx.slot_commit_file(descs[k][1], sizes[k]) as s:
                    assert roots[k] == s.root, k
        # the oracle: first and last slot of each batch, the whole slots, every member that is not synthetic
        check = sorted({b[0] for b in batches} | {b[-1] for b in batches} | set(whole) | {k for k, m in enumerate(members) if m[0] not in ("syn", "keep")})
        for k in check:
            if members[k][0] == "fake":
                want = orc.commit_fake_slot(descs[k][1], sizes[k] // CELL, n_threads=8)[0]
            else:
                data = host_bytes[k] if k in host_bytes else synthetic_ref(descs[k][1], 0, sizes[k])
                want = orc.commit_slot((data.ctypes.data, sizes[k]), n_threads=8)[0]
            assert roots[k] == want, (k, members[k])
        # the dataset tree and every slot's proof in it
        layers = orc.merkle_layers(roots)
        assert ds.root == layers[-1][0]
        depth = len(layers) - 1
        for k in range(n):
            want = [layers[i][(k >> i) ^ 1] if (k >> i) ^ 1 < len(layers[i]) else 0 for i in range(depth)] + [0] * (12 - depth)
            assert ds.slot_proof(k, 12) == want, k
        # the kept slot answers a challenge like the same slot committed alone, and every path reconstructs in two stages
        idx, paths, leaves = ds.prove(0xBEEF, 24, 32)
        with BorrowedSlot(pkg, ctx, ctx.lib.cdx_dataset_kept_slot(ds.h)) as kept:
            assert kept.root == roots[keep]
            (i2,), (p2,), (l2,) = kept.prove_batch([0xBEEF], 24, 32)
            assert (idx, paths, leaves) == (i2, p2, l2)
        assert idx == [orc.cell_index(0xBEEF, roots[keep], 16 * 32, c) for c in range(1, 25)]
        for ci, path, leaf in zip(idx, paths, leaves):
            blk = orc.reconstruct_root(leaf, ci % 32, 32, path[:5])
            assert orc.reconstruct_root(blk, ci // 32, 16, path[5:9]) == roots[keep]
            assert all(v == 0 for v in path[9:])


@pytest.mark.gpu
def test_dataset_launches_match_restatement(pkg, capi, ctx, torch_mod):
    """the same mix from host memory only, on a context whose pinned pipeline always starts the same way: the dataset
    commit launches exactly the kernels of its batches, of its whole slots committed alone and of the dataset tree"""
    torch = torch_mod
    members, keep = big_mix()
    sizes = [b * BLOCK for _, b, _ in members]
    whole, batches = partition(plan_dataset([b for _, b, _ in members], 1, BLOCK)[1][0], sizes, keep)
    d = torch.empty(sum(sizes), dtype=torch.uint8, device="cuda")
    ctx.fill_synthetic_dev(0xD00D, 0, d.numel(), d.data_ptr())
    host = d.cpu().numpy()
    del d
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + s)
    parts = [host[offs[k]:offs[k + 1]] for k in range(len(sizes))]
    c = fresh_context(pkg, CODEX_COMMIT_RAMP=0)
    try:
        alone = []
        for k in whole:
            before = c.launches
            with c.slot_commit_host(parts[k]) as s:
                alone.append(c.launches - before)
        want = sum(batch_launches([sizes[k] // BLOCK for k in b], BLOCK // CELL) for b in batches) + sum(alone) + tree_launches(len(sizes))
        before = c.launches
        with c.dataset_commit(None, [(capi.SRC_HOST, parts[k], sizes[k]) for k in range(len(sizes))], CELL, BLOCK, keep_slot=keep) as ds:
            got = c.launches - before
            roots = ds.slot_roots
        assert got == want, (got, want, len(batches))
        for k in (batches[0][0], batches[0][-1], batches[1][0], batches[1][-1], keep):
            with c.slot_commit_host(parts[k]) as s:
                assert roots[k] == s.root, k
    finally:
        c.close()


# ---- many trees in one segmented pass ----------------------------------------------------------------------------------

SEG_GEOMETRIES = [(64, 1, 20000), (64, 2, 4097), (64, 4, 4097), (36, 1, 4097), (36, 2, 4097), (36, 4, 20000)]


def draw_blocks(rnd, n):
    """block counts 1 .. 70, weighted toward one and two blocks: the trees of one batch reach their roots at different levels"""
    return [rnd.choice((1, 1, 1, 2, 2)) if rnd.random() < 0.6 else rnd.randint(3, 70) for _ in range(n)]


@pytest.mark.gpu
@pytest.mark.parametrize("cell,cpb,n_max", SEG_GEOMETRIES, ids=[f"cell{c}-cpb{k}" for c, k, _ in SEG_GEOMETRIES])
def test_segmented_pass_many_trees_vs_oracle(ctx, capi, orc, torch_mod, cell, cpb, n_max):
    """1, 255, 257, 4097 and (for one TMA and one plain-load geometry) 20 000 slots in one call, through the device and
    host batch entry points and a dataset of host-memory members; every root against the oracle.  The slot sets are
    prefixes of one draw, so the oracle roots are computed once."""
    torch = torch_mod
    block = cell * cpb
    rnd = random.Random(cell * 100 + cpb)
    blocks = draw_blocks(rnd, n_max)
    sizes = [b * block for b in blocks]
    host = random_bytes(cell + cpb, sum(sizes))
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + s)
    parts = [host[offs[k]:offs[k + 1]] for k in range(n_max)]
    want = oracle_roots(orc, parts, cell, block)
    dev = torch.from_numpy(host).cuda()
    for n in (1, 255, 257, 4097, 20000):
        if n > n_max:
            continue
        assert ctx.slots_commit_batch_dev(dev.data_ptr(), sizes[:n], cell, block) == want[:n], n
        assert ctx.slots_commit_batch_host(host, sizes[:n], cell, block) == want[:n], n
        with ctx.dataset_commit(None, [(capi.SRC_HOST, parts[k], sizes[k]) for k in range(n)], cell, block) as ds:
            assert ds.stats["batched"] == n
            assert ds.slot_roots == want[:n], n


@pytest.mark.gpu
def test_one_cell_slots_two_to_the_17(ctx, orc):
    """2^17 slots of one one-cell block in one batch: slot root = compress(compress(cell hash, 0, key 3), 0, key 3) (the
    block tree and the slot tree of one leaf), computed by two independent GPU calls; a sample against the oracle"""
    n, cell = 1 << 17, 64
    data = random_bytes(17, n * cell)
    roots = ctx.slots_commit_batch_host(data, [cell] * n, cell, cell)
    h = ctx.hash_bytes_batch(data.tobytes(), n, cell)
    blk = ctx.compress_batch(h, [0] * n, [3] * n)
    assert roots == ctx.compress_batch(blk, [0] * n, [3] * n)
    rnd = random.Random(17)
    picks = sorted(set(rnd.sample(range(n), 4096)) | {m + d for m in range(0, n + 1, 256) for d in (-1, 0, 1) if 0 <= m + d < n})
    want = oracle_roots(orc, [data[k * cell:(k + 1) * cell] for k in picks], cell, cell)
    assert [roots[k] for k in picks] == want


@pytest.mark.gpu
def test_batch_fake_300_seeds_vs_oracle(ctx, orc):
    rnd = random.Random(300)
    seeds = [0, 1, 2**64 - 1, 2**63] + [rnd.getrandbits(64) for _ in range(296)]
    roots = ctx.slots_commit_batch_fake(seeds, 12, 256, 1024)                  # three blocks of four 256-byte cells
    with cf.ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        want = list(ex.map(lambda s: orc.commit_fake_slot(s, 12, 256, 1024)[0], seeds))
    assert roots == want


# ---- synthetic bytes at any offset ------------------------------------------------------------------------------------

OFFSET_GEOMETRIES = [(100, 1), (100, 2), (36, 1), (36, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("cell,cpb", OFFSET_GEOMETRIES, ids=[f"cell{c}-cpb{k}" for c, k in OFFSET_GEOMETRIES])
def test_synthetic_members_behind_host_members(ctx, capi, orc, cell, cpb):
    """synthetic members whose place in the batch buffer (the sum of the sizes before them in LPT order) or whose own size
    is not a multiple of 8: every root equals the oracle over the byte-exact definition"""
    block = cell * cpb
    kinds = [("host", 3), ("syn", 7), ("host", 1), ("syn", 5), ("syn", 3), ("host", 9), ("syn", 1), ("syn", 11), ("host", 13)]
    sizes = [b * block for _, b in kinds]
    data, descs = [], []
    for k, (kind, _) in enumerate(kinds):
        if kind == "host":
            data.append(random_bytes(k, sizes[k]))
            descs.append((capi.SRC_HOST, data[-1], sizes[k]))
        else:
            data.append(synthetic_ref(0x0FF5E7 + k, 0, sizes[k]))
            descs.append((capi.SRC_SYNTHETIC, 0x0FF5E7 + k, sizes[k]))
    _, batches = partition(plan_dataset([b for _, b in kinds], 1, block)[1][0], sizes)
    off, odd = 0, 0
    for k in batches[0]:
        odd += kinds[k][0] == "syn" and (off % 8 != 0 or sizes[k] % 8 != 0)
        off += sizes[k]
    assert odd >= (3 if block % 8 else 0)
    with ctx.dataset_commit(None, descs, cell, block) as ds:
        assert ds.stats["batched"] == len(kinds)
        assert ds.slot_roots == oracle_roots(orc, data, cell, block)


@pytest.mark.gpu
def test_synthetic_tiles_starting_inside_a_word(pkg, capi, ctx, orc, torch_mod):
    """a whole synthetic slot of 36-byte one-cell blocks over three 16 MiB tiles: a tile is 466 033 blocks (16 777 188
    bytes), so the second tile starts 4 bytes into a word.  Root and every cell hash equal the resident commit of the
    reference bytes, and the oracle's root"""
    torch = torch_mod
    cell, tile_blocks = 36, (16 << 20) // 36
    n_blocks = 2 * tile_blocks + 300001                                      # odd: the slot ends inside a word too
    n = n_blocks * cell
    assert (tile_blocks * cell) % 8 == 4 and n % 8 == 4
    ref = synthetic_ref(0x711E, 0, n)
    dev = torch.from_numpy(ref).cuda()
    c = fresh_context(pkg, CODEX_COMMIT_TILE_MIB=16)
    try:
        with c.dataset_commit(None, [(capi.SRC_SYNTHETIC, 0x711E, n)], cell, cell, keep_slot=0) as ds, \
                BorrowedSlot(pkg, c, c.lib.cdx_dataset_kept_slot(ds.h)) as kept, ctx.slot_commit_dev(dev.data_ptr(), n, cell, cell) as resident:
            assert ds.stats["whole"] == 1
            assert kept.root == resident.root == ds.slot_roots[0]
            assert raw_layer(c, kept.h, 0, 0, 0, n_blocks) == raw_layer(ctx, resident.h, 0, 0, 0, n_blocks)
            assert kept.root == orc.commit_slot((ref.ctypes.data, n), cell, cell, n_threads=8)[0]
    finally:
        c.close()


@pytest.mark.gpu
def test_synthetic_slot_leaves_no_byte_unwritten(ctx, capi, orc):
    """a synthetic slot of three 100-byte blocks (300 bytes: the last 4 are half a word) committed, then a different slot
    of junk bytes into the same pooled buffer, then the first again: both roots are the oracle's"""
    ref = synthetic_ref(0x7A11, 0, 300)
    want = orc.commit_slot((ref.ctypes.data, 300), 100, 100)[0]
    junk = random_bytes(5, 4000)
    roots = []
    for descs in ([(capi.SRC_SYNTHETIC, 0x7A11, 300)], [(capi.SRC_HOST, junk, 4000)], [(capi.SRC_SYNTHETIC, 0x7A11, 300)]):
        with ctx.dataset_commit(None, descs, 100, 100) as ds:
            roots.append(ds.slot_roots[0])
    assert roots[0] == roots[2] == want
    assert roots[1] == orc.commit_slot((junk.ctypes.data, 4000), 100, 100)[0]
