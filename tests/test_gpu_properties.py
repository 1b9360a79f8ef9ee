"""GPU tests at sizes the oracle cannot re-hash in seconds: size-independent properties of the commitment
(sharded == unsharded, tiled host path == resident path, tree of read-back block hashes == root, every sampled path
reconstructs in two stages), plus the single-GPU emulation of the multi-rank exchange through the C ABI."""
import importlib
import random

import pytest

from conftest import PKG

pytestmark = pytest.mark.gpu
R = 21888242871839275222246405745257275088548364400416034343698204186575808495617


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def synthetic(ctx, torch, n_bytes, seed=0xC0DE, first_word=0):
    d = torch.empty(n_bytes, dtype=torch.uint8, device="cuda")
    ctx.fill_synthetic_dev(seed, first_word, n_bytes, d.data_ptr())
    torch.cuda.synchronize()
    return d


def install_top(torch, shards):
    """single-GPU stand-in for the NCCL exchange inside cdx_slot_exchange_top: concatenate the level-T nodes of the
    emulated ranks (low-level ABI: cdx_slot_subtree_roots_copy_dev) and install them on each (cdx_slot_set_top_dev)"""
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


def commit_in_ranges(ctx, torch, sharded, d, n_blocks, ranges, top_level):
    """what N ranks do, run back to back on one GPU: per-range commit, exchange of the level-T nodes, replicated top"""
    shards = []
    for first, count in ranges:
        if count == 0:
            shards.append(None)
            continue
        ptr = d.data_ptr() + first * 65536
        shards.append(ctx.slot_commit_range_dev(ptr, count * 65536, 2048, 65536, first, n_blocks, top_level))
    gathered = install_top(torch, [s for s in shards if s is not None])
    assert gathered.numel() == 32 * sharded.level_width(n_blocks, top_level)
    return shards


@pytest.mark.parametrize("n_blocks,world", [(16384, 4), (1000, 3), (163, 8), (25 * 64, 8)])
def test_sharded_commit_equals_whole_commit(ctx, torch_mod, n_blocks, world):
    torch = torch_mod
    sharded = importlib.import_module(PKG + ".sharded")
    d = synthetic(ctx, torch, n_blocks * 65536)
    with ctx.slot_commit_dev(d.data_ptr(), n_blocks * 65536) as whole:
        root = whole.root
        top_level, ranges = sharded.plan_block_ranges(n_blocks, world, max_imbalance=0.05)
        assert importlib.import_module(PKG).capi.block_ranges_top_level(n_blocks, ranges) >= top_level   # the library accepts this plan
        shards = commit_in_ranges(ctx, torch, sharded, d, n_blocks, ranges, top_level)
        live = [s for s in shards if s is not None]
        assert all(s.root == root for s in live)
        # paths: the owner produces the whole path, everyone else zeros -> the SUM over ranks is the path
        rnd = random.Random(n_blocks)
        cells = [rnd.randrange(32 * n_blocks) for _ in range(20)] + [0, 32 * n_blocks - 1]
        ref_paths, ref_leaves = whole.cell_paths(cells, 32)
        acc = [[0] * 32 for _ in cells]
        acc_leaf = [0] * len(cells)
        for s in live:
            p, l = s.cell_paths(cells, 32)
            for i in range(len(cells)):
                acc[i] = [a + b for a, b in zip(acc[i], p[i])]
                acc_leaf[i] += l[i]
        assert acc == ref_paths and acc_leaf == ref_leaves
        for s in live:
            s.free()


def test_one_gib_slot_properties(ctx, orc, torch_mod):
    torch = torch_mod
    n_blocks = 16384
    d = synthetic(ctx, torch, n_blocks * 65536)
    with ctx.slot_commit_dev(d.data_ptr(), n_blocks * 65536) as slot:
        n_cells, nb, bd, sd = slot.shape
        assert (n_cells, nb, bd, sd) == (524288, 16384, 5, 14)
        root = slot.root
        # a checksum of checksums: the tree over the read-back block hashes is the root (GPU tree API and oracle)
        bh = slot.read_layer(1, 0, 0, n_blocks)
        assert ctx.merkle_root(bh) == root == orc.merkle_root(bh)
        # spot-check cell hashes and one block tree against the oracle
        host = d[: 2 * 65536].cpu().numpy().tobytes()
        assert slot.read_layer(0, 0, 0, 64) == [orc.hash_bytes(host[i * 2048:(i + 1) * 2048]) for i in range(64)]
        tail = d[(n_blocks - 1) * 65536:].cpu().numpy().tobytes()
        assert slot.read_layer(1, 0, n_blocks - 1, 1)[0] == orc.merkle_root([orc.hash_bytes(tail[i * 2048:(i + 1) * 2048]) for i in range(32)])
        # 100 sampled paths (BASELINE config 5 shape) all reconstruct to the root in two stages (Slot.hs:189-217)
        idx = ctx.cell_indices(987654321, root, n_cells, 100)
        assert idx == [orc.cell_index(987654321, root, n_cells, c) for c in range(1, 101)]
        paths, leaves = slot.cell_paths(idx, 32)
        for i, p, leaf in zip(idx, paths, leaves):
            blk = orc.reconstruct_root(leaf, i % 32, 32, p[:5])
            assert orc.reconstruct_root(blk, i // 32, n_blocks, p[5:19]) == root
            assert all(v == 0 for v in p[19:])
    # the tiled host-buffer path (4 x 256 MiB tiles, copy overlapped with the sponge) gives the same root
    host_all = d.cpu().numpy()
    with ctx.slot_commit_host(host_all) as slot2:
        assert slot2.root == root
    # the same bytes from pinned memory (direct async copies instead of the pinned-chunk pipeline pageable memory takes)
    pinned = torch.empty(n_blocks * 65536, dtype=torch.uint8, pin_memory=True)
    pinned.copy_(d)
    torch.cuda.synchronize()
    with ctx.slot_commit_host(pinned.data_ptr(), n_bytes=n_blocks * 65536) as slot3:
        assert slot3.root == root
    # two ranks' worth of pageable host ranges (512 MiB each: the chunk pipeline with a non-zero first block), exchanged
    sharded = importlib.import_module(PKG + ".sharded")
    half = n_blocks // 2
    shards = [ctx.slot_commit_range_host(host_all[k * half * 65536:(k + 1) * half * 65536], 2048, 65536, k * half, n_blocks, 13)
              for k in range(2)]
    install_top(torch, shards)
    assert [s.root for s in shards] == [root, root]
    for s in shards:
        s.free()


def test_idempotence_and_sensitivity(ctx, torch_mod):
    torch = torch_mod
    n = 300 * 65536
    d = synthetic(ctx, torch, n)
    with ctx.slot_commit_dev(d.data_ptr(), n) as a, ctx.slot_commit_dev(d.data_ptr(), n) as b:
        assert a.root == b.root
        ra = a.root
    d[n - 1] ^= 1                                                    # flip one bit of the very last byte
    torch.cuda.synchronize()
    with ctx.slot_commit_dev(d.data_ptr(), n) as c:
        assert c.root != ra


def test_permutation_batch_2_20_vs_oracle(ctx, orc, torch_mod):
    """BASELINE config 2 at its full size (SURVEY.md 8d): 2^20 states, the first 2^19 are (j, j+1, j+2) -- state 0 is the
    stored KAT input (Example.hs:13-22) -- the rest arbitrary 256-bit values (taken mod r); every output element is
    compared with the oracle (multi-threaded over the batch)"""
    import concurrent.futures as cf
    import numpy as np
    torch = torch_mod
    n, half = 1 << 20, 1 << 19
    a = synthetic(ctx, torch, 96 * n, seed=1)
    host = a.cpu().numpy().copy()
    small = np.zeros((half, 3, 4), dtype=np.uint64)
    j = np.arange(half, dtype=np.uint64)
    for k in range(3):
        small[:, k, 0] = j + np.uint64(k)
    host[:96 * half] = small.reshape(-1).view(np.uint8)
    a.copy_(torch.from_numpy(host))
    b = torch.empty_like(a)
    ctx.permutation_batch_dev(a.data_ptr(), b.data_ptr(), n)
    torch.cuda.synchronize()
    out = b.cpu().numpy().tobytes()
    inp = host.tobytes()
    kat = [0x30610a447b7dec194697fb50786aa7421494bd64c221ba4d3b1af25fb07bd103, 0x13f731d6ffbad391be22d2ac364151849e19fa38eced4e761bcd21dbdc600288,
           0x1433e2c8f68382c447c5c14b8b3df7cbfd9273dd655fe52f1357c27150da786f]                      # Example.hs:17-21
    assert [int.from_bytes(out[32 * k:32 * k + 32], "little") for k in range(3)] == kat
    chunk = 96 * (1 << 16)
    with cf.ThreadPoolExecutor(8) as ex:                                     # ctypes releases the GIL inside the oracle
        parts = list(ex.map(lambda o: orc.permutation_batch_bytes(inp[o:o + chunk]), range(0, len(inp), chunk)))
    assert b"".join(parts) == out


def test_dataset_commit_small_vs_oracle(ctx, orc, torch_mod):
    """BASELINE config 5 in miniature through cdx_dataset_commit: 13 slots of mixed size (odd nodes in the dataset tree;
    the small ones go through the batched path, the kept one is committed whole), slot 3 sampled"""
    import bench
    dataset = importlib.import_module(PKG + ".dataset")
    blocks = dataset.draw_slot_blocks(13, 3 * 65536, 40 * 65536, seed=99, pow2_slot=3, pow2_blocks=16)
    assert blocks[3] == 16 and len(set(blocks)) > 5
    with ctx.dataset_commit(None, dataset.synthetic_descs(blocks, 99), keep_slot=3) as ds:
        roots = ds.slot_roots
        assert ds.stats["batched"] == 12 and ds.stats["whole"] == 1 and ds.stats["bytes_local"] == sum(blocks) * 65536
        # every slot root against the oracle over the same synthetic bytes (bench.py's numpy twin of the device generator)
        for k in range(13):
            data = bench.synthetic_bytes_host(dataset.slot_seed(99, k), 0, blocks[k] * 65536)
            root, _, _ = orc.commit_slot((data.ctypes.data, blocks[k] * 65536), n_threads=4)
            assert roots[k] == root, k
        layers = orc.merkle_layers(roots)
        assert ds.root == layers[-1][0]
        proof = ds.slot_proof(3, 8)
        assert orc.reconstruct_root(roots[3], 3, 13, proof[:len(layers) - 1]) == ds.root
        assert proof[len(layers) - 1:] == [0] * (8 - (len(layers) - 1))
        for k in (0, 12):
            assert orc.reconstruct_root(roots[k], k, 13, ds.slot_proof(k, 8)[:len(layers) - 1]) == ds.root
        n_cells = 16 * 32
        idx, paths, leaves = ds.prove(1234567, 20, 32)
        assert idx == [orc.cell_index(1234567, roots[3], n_cells, c) for c in range(1, 21)]
        for ci, path, leaf in zip(idx, paths, leaves):
            blk = orc.reconstruct_root(leaf, ci % 32, 32, path[:5])
            assert orc.reconstruct_root(blk, ci // 32, 16, path[5:9]) == roots[3]
            assert all(v == 0 for v in path[9:])
    bins = dataset.lpt_assign(blocks, 4)
    assert sorted(k for b in bins for k in b) == list(range(13))
    loads = [sum(blocks[k] for k in b) for b in bins]
    assert max(loads) <= 1.34 * sum(blocks) / 4


def test_dataset_commit_mixed_sources(ctx, orc, torch_mod, tmp_path):
    """every slot source kind in one dataset: the reference's fake data, synthetic bytes, a file, host memory; big enough
    slots (> 64 MiB) take the whole-slot path, the rest the batched one; roots equal the single-slot entry points"""
    import numpy as np
    import bench
    capi = importlib.import_module(PKG).capi
    small, big = 5 * 65536, 1100 * 65536                                   # 320 KiB (batched) and 68.75 MiB (whole)
    host_small = bench.synthetic_bytes_host(11, 0, small).copy()
    host_big = bench.synthetic_bytes_host(12, 0, big).copy()
    f_small, f_big = str(tmp_path / "s.dat"), str(tmp_path / "b.dat")
    bench.synthetic_bytes_host(13, 0, small).tofile(f_small)
    bench.synthetic_bytes_host(14, 0, big).tofile(f_big)
    descs = [(capi.SRC_FAKE, 4242, small), (capi.SRC_SYNTHETIC, 15, small), (capi.SRC_FILE, f_small, small), (capi.SRC_HOST, host_small, small),
             (capi.SRC_SYNTHETIC, 16, big), (capi.SRC_FILE, f_big, big), (capi.SRC_HOST, host_big, big), (capi.SRC_FAKE, 4243, 65536)]
    with ctx.dataset_commit(None, descs) as ds:
        roots = ds.slot_roots
        assert ds.stats == {"bytes_local": 4 * small + 3 * big + 65536, "whole": 3, "batched": 5, "sharded": 0}
    with ctx.slot_commit_fake(4242, small // 2048) as s:
        assert roots[0] == s.root == orc.commit_fake_slot(4242, small // 2048)[0]
    for k, seed in ((1, 15), (4, 16)):
        data = bench.synthetic_bytes_host(seed, 0, descs[k][2])
        assert roots[k] == orc.commit_slot((data.ctypes.data, descs[k][2]), n_threads=8)[0]
    with ctx.slot_commit_file(f_small, small) as s:
        assert roots[2] == s.root
    with ctx.slot_commit_host(host_small) as s:
        assert roots[3] == s.root
    with ctx.slot_commit_file(f_big, big) as s:
        assert roots[5] == s.root
    with ctx.slot_commit_host(host_big) as s:
        assert roots[6] == s.root
    assert roots[7] == orc.commit_fake_slot(4243, 32)[0]                     # a one-block slot: key-3 singleton rule
    with pytest.raises(Exception):
        ctx.dataset_commit(None, [(capi.SRC_FILE, str(tmp_path / "missing.dat"), small)])


def test_commit_from_file(ctx, torch_mod, tmp_path):
    """SlotFile at speed (SURVEY.md 8f.1): pread -> pinned -> H2D -> sponge; equals the resident commitment; a short file
    reads as zeros past its end (slot.nim:64-65); offsets select a window"""
    import time
    torch = torch_mod
    n = 700 * 65536                                                      # 43.75 MiB ... plus a multi-tile case below
    d = synthetic(ctx, torch, n)
    host = d.cpu().numpy()
    path = str(tmp_path / "slot.dat")
    host.tofile(path)
    with ctx.slot_commit_dev(d.data_ptr(), n) as a, ctx.slot_commit_file(path, n) as b:
        assert a.root == b.root
    short = 600 * 65536 + 1234
    host[:short].tofile(path)
    padded = host.copy()
    padded[short:] = 0
    with ctx.slot_commit_host(padded) as a, ctx.slot_commit_file(path, n) as b:
        assert a.root == b.root
    host.tofile(path)
    with ctx.slot_commit_dev(d.data_ptr() + 100 * 65536, 64 * 65536) as a, ctx.slot_commit_file(path, 64 * 65536, offset=100 * 65536) as b:
        assert a.root == b.root
    big = 9 * 1024 * 65536 + 3 * 65536                                  # 579 MiB: three device tiles, ten pinned chunks, ragged tail
    d2 = synthetic(ctx, torch, big, seed=7)
    path2 = str(tmp_path / "big.dat")
    d2.cpu().numpy().tofile(path2)
    with ctx.slot_commit_dev(d2.data_ptr(), big) as a:
        ra = a.root
    t0 = time.perf_counter()
    with ctx.slot_commit_file(path2, big) as b:
        dt = time.perf_counter() - t0
        assert b.root == ra
    print(f"commit_file {big / 2**20:.0f} MiB from page cache: {big / dt / 1e9:.2f} GB/s")


def test_commit_file_vs_oracle(ctx, orc, torch_mod, tmp_path):
    """the file path against the ORACLE on the same bytes (not against another CUDA path): whole file, short file
    (zero-filled tail, slot.nim:64-65) and an offset window"""
    import bench
    n = 300 * 65536
    data = bench.synthetic_bytes_host(0xF11E, 0, n).copy()
    path = str(tmp_path / "slot.dat")
    data.tofile(path)
    with ctx.slot_commit_file(path, n) as s:
        assert s.root == orc.commit_slot((data.ctypes.data, n), n_threads=8)[0]
    short = 250 * 65536 + 777
    data[:short].tofile(path)
    padded = data.copy()
    padded[short:] = 0
    with ctx.slot_commit_file(path, n) as s:
        assert s.root == orc.commit_slot((padded.ctypes.data, n), n_threads=8)[0]
    data.tofile(path)
    win = data[70 * 65536:(70 + 33) * 65536].copy()
    with ctx.slot_commit_file(path, 33 * 65536, offset=70 * 65536) as s:
        assert s.root == orc.commit_slot((win.ctypes.data, 33 * 65536), n_threads=8)[0]
    with pytest.raises(Exception):
        ctx.slot_commit_file(str(tmp_path / "nope.dat"), n)


def test_ten_gib_slot_random_blocks_vs_oracle(ctx, orc, torch_mod):
    """BASELINE config 3 at full size: 64 random blocks spread over the whole 10 GiB slot (so offsets far above 4 GiB, where
    32-bit row or byte arithmetic would wrap) are re-hashed by the oracle from the same bytes and compared with the block
    hashes and cell hashes the GPU retained; the root must be the oracle's tree over the GPU's block hashes, and the
    known 10 GiB root of this seed"""
    torch = torch_mod
    n_blocks = 163840
    d = synthetic(ctx, torch, n_blocks * 65536)
    with ctx.slot_commit_dev(d.data_ptr(), n_blocks * 65536) as slot:
        root = slot.root
        rnd = random.Random(10)
        picks = sorted({0, n_blocks - 1, 65536, 65537, 131071} | {rnd.randrange(n_blocks) for _ in range(59)})
        assert max(picks) * 65536 > (9 << 30)
        for b in picks:
            raw = d[b * 65536:(b + 1) * 65536].cpu().numpy().tobytes()
            cells = [orc.hash_bytes(raw[i * 2048:(i + 1) * 2048]) for i in range(32)]
            assert slot.read_layer(0, 0, 32 * b, 32) == cells, b
            assert slot.read_layer(1, 0, b, 1)[0] == orc.merkle_root(cells), b
        bh = slot.read_layer(1, 0, 0, n_blocks)
        assert orc.merkle_root(bh) == root
    del d
    torch.cuda.empty_cache()


def test_batched_small_slots(ctx, orc, torch_mod):
    """cdx_slots_commit_batch_*: many slots in one pass == each slot committed alone == the oracle; ragged block counts
    (odd nodes per slot), one-block slots (singleton rule), and the reference's fake data with per-slot seeds"""
    import bench
    torch = torch_mod
    blocks = [64, 1, 3, 2, 7, 1, 33, 64, 5, 100, 1, 16]
    sizes = [b * 65536 for b in blocks]
    total = sum(sizes)
    d = synthetic(ctx, torch, total, seed=77)
    roots = ctx.slots_commit_batch_dev(d.data_ptr(), sizes)
    host = d.cpu().numpy()
    off = 0
    for k, sz in enumerate(sizes):
        part = host[off:off + sz].copy()
        with ctx.slot_commit_dev(d.data_ptr() + off, sz) as s:
            assert roots[k] == s.root, k
        assert roots[k] == orc.commit_slot((part.ctypes.data, sz), n_threads=4)[0], k
        off += sz
    assert ctx.slots_commit_batch_host(host, sizes) == roots
    # config 1's eleven slots (seed 12345 + 72 + 1001 k, 64 blocks each) in one call
    seeds = [12345 + 72 + 1001 * k for k in range(11)]
    fr = ctx.slots_commit_batch_fake(seeds, 2048)
    assert fr[3] == 16142339001376051487701717049451130483290782524159378806355159917477338192952   # SURVEY.md 8c, config 1 slotRoot
    for k in (0, 10):
        assert fr[k] == orc.commit_fake_slot(seeds[k], 2048, n_threads=4)[0]
    assert ctx.merkle_root(fr) == 7410604474820069305866101106843319395502234157925946588762357169176803727431      # config 1 dataSetRoot
    # other geometry: one-cell blocks and 8-cell blocks
    for cell, block, bl in ((128, 128, [1, 2, 5]), (256, 2048, [3, 1, 8])):
        sz = [b * block for b in bl]
        dd = synthetic(ctx, torch, sum(sz), seed=5)
        rr = ctx.slots_commit_batch_dev(dd.data_ptr(), sz, cell, block)
        o = 0
        for k, z in enumerate(sz):
            with ctx.slot_commit_dev(dd.data_ptr() + o, z, cell, block) as s:
                assert rr[k] == s.root
            o += z
    with pytest.raises(Exception):
        ctx.slots_commit_batch_dev(d.data_ptr(), [65536, 1000])


def test_sharded_entry_points_single_rank(ctx, torch_mod):
    """cdx_slot_commit_sharded_* / cdx_slot_cell_paths_sharded / cdx_slot_prove_batch_sharded with a one-rank communicator
    (no NCCL involved) equal the whole-slot entry points"""
    torch = torch_mod
    n_blocks = 1024
    d = synthetic(ctx, torch, n_blocks * 65536, seed=3)
    comm = ctx.comm_init(1, 0, None)
    assert (comm.rank, comm.size) == (0, 1)
    comm.barrier()
    with ctx.slot_commit_dev(d.data_ptr(), n_blocks * 65536) as whole:
        for T in (0, 4, 10):
            with ctx.slot_commit_sharded_dev(comm, d.data_ptr(), n_blocks * 65536, 2048, 65536, 0, n_blocks, T) as sh:
                assert sh.root == whole.root
                cells = [0, 5, 32767, 12345]
                assert sh.cell_paths_sharded(comm, cells, 32) == whole.cell_paths(cells, 32)
                assert sh.prove_batch_sharded(comm, [1, 2, 3], 7, 32) == whole.prove_batch([1, 2, 3], 7, 32)
        host = d.cpu().numpy()
        with ctx.slot_commit_sharded_host(comm, host, n_blocks * 65536, 2048, 65536, 0, n_blocks, 6) as sh:
            assert sh.root == whole.root
    comm.destroy()


def _nccl_rank(rank, world, id_q, out_q, n_blocks, extra=None):
    """one process per GPU: the library's own communicator (the id travels through a multiprocessing queue -- no
    torch.distributed anywhere), sharded commit, collective paths, dataset commit"""
    import importlib as il
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    pkg = il.import_module("codex-storage-proofs-circuits_b200")
    dataset = il.import_module("codex-storage-proofs-circuits_b200.dataset")
    torch.cuda.set_device(rank)
    ctx = pkg.Context(rank)
    if rank == 0:
        uid = pkg.capi.comm_unique_id()
        for _ in range(world - 1):
            id_q.put(uid)
    else:
        uid = id_q.get(timeout=120)
    comm = ctx.comm_init(world, rank, uid)
    res = {}
    for nb in n_blocks:
        T, ranges = pkg.capi.plan_block_ranges(nb, world)
        first, count = ranges[rank]
        d = torch.empty(max(count, 1) * 65536, dtype=torch.uint8, device="cuda")
        if count:
            ctx.fill_synthetic_dev(0xC0DE, first * 8192, count * 65536, d.data_ptr())
        sh = ctx.slot_commit_sharded_dev(comm, d.data_ptr(), count * 65536, 2048, 65536, first, nb, T)
        cells = sorted({0, 32 * nb - 1, 16 * nb, 32 * (nb // 2) + 7})
        paths, leaves = sh.cell_paths_sharded(comm, cells, 32)
        res[nb] = (sh.root, T, ranges, cells, paths, leaves)
        if nb & (nb - 1) == 0:
            res[(nb, "prove")] = sh.prove_batch_sharded(comm, [11, 12], 5, 32)
        host = d.cpu().numpy()
        sh2 = ctx.slot_commit_sharded_host(comm, host, count * 65536, 2048, 65536, first, nb, T)
        assert sh2.root == sh.root
        sh.free(); sh2.free()
    # dataset: 9 slots, one big enough to be sharded over the ranks (>= 256 MiB per rank), slot 2 kept
    blocks = [40, 8192 * world, 64, 7, 300, 1, 1200, 33, 2]
    ds = ctx.dataset_commit(comm, dataset.synthetic_descs(blocks, 5), keep_slot=2)
    res["dataset"] = (ds.root, ds.slot_roots, ds.stats, ds.prove(99, 10, 32), ds.slot_proof(2, 8))
    ds.free()
    ds = ctx.dataset_commit(comm, dataset.synthetic_descs([16384 * world, 5], 6), keep_slot=0)   # the kept slot is the sharded one
    res["dataset_sharded_keep"] = (ds.root, ds.slot_roots, ds.stats, ds.prove(7, 6, 32))
    ds.free()
    # sharded members that are NOT generated: a file (each rank preads its own block range) and host memory (each rank
    # copies its own range); both are big enough (256 MiB per rank) to be sharded
    if extra is not None:
        import numpy as np
        path, n_bytes = extra
        host = np.fromfile(path, dtype=np.uint8)
        ds = ctx.dataset_commit(comm, [(pkg.capi.SRC_FILE, path, n_bytes), (pkg.capi.SRC_HOST, host, n_bytes), (pkg.capi.SRC_SYNTHETIC, 9, 65536)], keep_slot=0)
        res["dataset_file_host"] = (ds.root, ds.slot_roots, ds.stats, ds.prove(3, 4, 32))
        ds.free()
    comm.destroy()
    ctx.close()
    out_q.put((rank, res))


def test_nccl_sharded_and_dataset_two_gpus(ctx, orc, torch_mod, tmp_path):
    """the NCCL path proper (skipped below 2 GPUs): two processes, two GPUs, the library's communicator; the sharded root,
    paths and proofs equal the whole-slot ones computed on one GPU, for a power-of-two slot, a ragged one and a one-block
    slot (rank 1 holds an EMPTY shard); the two-rank dataset equals the one-rank dataset"""
    torch = torch_mod
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    dataset = importlib.import_module(PKG + ".dataset")
    world, n_blocks = 2, [4096, 1000, 1]
    mpc = mp.get_context("spawn")
    id_q, out_q = mpc.Queue(), mpc.Queue()
    big = 8192 * world * 65536                                              # 1 GiB: 512 MiB per rank, a power-of-two cell count
    big_path = str(tmp_path / "big_slot.dat")
    big_dev = synthetic(ctx, torch, big, seed=21)
    big_dev.cpu().numpy().tofile(big_path)
    procs = [mpc.Process(target=_nccl_rank, args=(r, world, id_q, out_q, n_blocks, (big_path, big))) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(out_q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for nb in n_blocks:
        d = synthetic(ctx, torch, nb * 65536)
        with ctx.slot_commit_dev(d.data_ptr(), nb * 65536) as whole:
            for r in range(world):
                root, T, ranges, cells, paths, leaves = results[r][nb]
                assert root == whole.root, (nb, r)
                assert (paths, leaves) == whole.cell_paths(cells, 32), (nb, r)
                if nb & (nb - 1) == 0:
                    assert results[r][(nb, "prove")] == whole.prove_batch([11, 12], 5, 32)
    assert sorted(c for _, c in results[0][1][2]) == [0, 1]                   # n_blocks = 1: one of the two ranks held an empty shard
    blocks = [40, 8192 * world, 64, 7, 300, 1, 1200, 33, 2]
    with ctx.dataset_commit(None, dataset.synthetic_descs(blocks, 5), keep_slot=2) as ds:
        one = (ds.root, ds.slot_roots, ds.prove(99, 10, 32), ds.slot_proof(2, 8))
    for r in range(world):
        root, roots, stats, proof, sproof = results[r]["dataset"]
        assert (root, roots, proof, sproof) == one, r
        assert stats["sharded"] == 1
    assert sum(results[r]["dataset"][2]["bytes_local"] for r in range(world)) == sum(blocks) * 65536
    with ctx.dataset_commit(None, dataset.synthetic_descs([16384 * world, 5], 6), keep_slot=0) as ds:
        one = (ds.root, ds.slot_roots, ds.prove(7, 6, 32))
    for r in range(world):
        root, roots, stats, proof = results[r]["dataset_sharded_keep"]
        assert (root, roots, proof) == one, r
    # file- and host-backed sharded members against the same bytes committed resident on one GPU
    with ctx.slot_commit_dev(big_dev.data_ptr(), big) as whole:
        (idx,), (paths,), (leaves,) = whole.prove_batch([3], 4, 32)
        for r in range(world):
            root, roots, stats, proof = results[r]["dataset_file_host"]
            assert roots[0] == roots[1] == whole.root, r
            assert stats["sharded"] == 2 and stats["bytes_local"] in (big, big + 65536)
            assert proof == (idx, paths, leaves), r


def test_fuzz_geometries_batch_dataset_and_single_agree_with_oracle(ctx, orc, torch_mod):
    """seeded fuzz over cell size (multiples of 4: both the TMA and the plain-load kernels), cells per block (powers of two
    incl. one-cell blocks), ragged slot sizes and batch composition: the batched entry point, the dataset commit and the
    single-slot commit must agree, and the oracle must agree with them on a slot of every case"""
    import bench
    capi = importlib.import_module(PKG).capi
    torch = torch_mod
    rnd = random.Random(20261018)
    for case in range(24):
        cell = rnd.choice([64, 96, 128, 160, 256, 388, 512, 1024, 2048, 2052, 4096])
        cpb = rnd.choice([1, 2, 4, 8, 32, 64])
        block = cell * cpb
        n_slots = rnd.randint(1, 9)
        blocks = [rnd.choice([1, 1, 2, 3, 5, 8, 13, 33, 64, 100]) for _ in range(n_slots)]
        sizes = [b * block for b in blocks]
        total = sum(sizes)
        d = synthetic(ctx, torch, (total + 7) // 8 * 8, seed=1000 + case)   # the fill writes whole 8-byte words
        roots = ctx.slots_commit_batch_dev(d.data_ptr(), sizes, cell, block)
        host = d.cpu().numpy()
        off, singles = 0, []
        for sz in sizes:
            if (d.data_ptr() + off) % 16 == 0:
                with ctx.slot_commit_dev(d.data_ptr() + off, sz, cell, block) as s:
                    singles.append(s.root)
            else:                                            # the device entry point wants a 16-byte aligned base
                with ctx.slot_commit_host(host[off:off + sz].copy(), cell, block) as s:
                    singles.append(s.root)
            off += sz
        assert roots == singles, (case, cell, cpb, blocks)
        k = rnd.randrange(n_slots)
        o = sum(sizes[:k])
        part = host[o:o + sizes[k]].copy()
        assert roots[k] == orc.commit_slot((part.ctypes.data, sizes[k]), cell, block, n_threads=4)[0], (case, cell, cpb, blocks, k)
        descs, o = [], 0
        for sz in sizes:
            descs.append((capi.SRC_HOST, host[o:o + sz].copy(), sz))
            o += sz
        keep = rnd.randrange(n_slots)
        with ctx.dataset_commit(None, descs, cell, block, keep_slot=keep) as ds:
            assert ds.slot_roots == roots, (case, cell, cpb, blocks)
            assert ds.root == orc.merkle_root(roots)
            n_cells = blocks[keep] * cpb
            if n_cells & (n_cells - 1) == 0 and n_cells > 1:
                idx, paths, leaves = ds.prove(case + 1, 3, 40)
                assert idx == [orc.cell_index(case + 1, roots[keep], n_cells, c) for c in range(1, 4)]


def test_cell_sponge_launch_boundary(pkg, ctx, torch_mod):
    """slots of more than 2^30 cells are hashed by several launches, each with its own tensor-map base (TMA row
    coordinates are signed 32-bit).  CODEX_COMMIT_MAX_LAUNCH_CELLS lowers that boundary for a fresh context so that a small
    slot crosses it several times, on the TMA path (64-byte cells) and on the plain-load path (100-byte cells): same roots,
    same cell hashes as the single-launch context"""
    import os
    torch = torch_mod
    cases = [(64, 64 * 32, 1000 * 32), (100, 100 * 8, 777 * 8), (2048, 65536, 300 * 32)]
    os.environ["CODEX_COMMIT_MAX_LAUNCH_CELLS"] = "4096"
    try:
        small = pkg.Context(0)
    finally:
        del os.environ["CODEX_COMMIT_MAX_LAUNCH_CELLS"]
    for cell, block, n_cells in cases:
        n_bytes = n_cells * cell
        d = synthetic(ctx, torch, (n_bytes + 7) // 8 * 8, seed=cell)
        with ctx.slot_commit_dev(d.data_ptr(), n_bytes, cell, block) as a, small.slot_commit_dev(d.data_ptr(), n_bytes, cell, block) as b:
            assert a.root == b.root, (cell, block)
            assert a.read_layer(0, 0, 0, n_cells) == b.read_layer(0, 0, 0, n_cells)
        host = d[:n_bytes].cpu().numpy()
        with small.slot_commit_host(host, cell, block) as c, ctx.slot_commit_host(host, cell, block) as e:
            assert c.root == e.root
    small.close()


def _tiles(n_blocks, wants):
    """number of tiles a schedule cuts n_blocks into: `wants` yields each tile's size, the last one is clipped"""
    done = n = 0
    for want in wants:
        if done >= n_blocks:
            return n
        done += min(want, n_blocks - done)
        n += 1


def _pinned_wants(n_bytes, block, tile_mib, gradual):
    n_blocks = n_bytes // block
    target = tile_mib << 20 if n_bytes >= 1 << 30 else max(n_bytes // 4, 16 << 20)
    tile = min(max(target // block, 1), n_blocks)
    if n_blocks > tile and tile >= 8:
        if gradual:
            cur = max(tile // 4, 1)
            while cur < tile:
                yield cur
                cur += max(cur // 4, 1)
        else:
            yield max(tile // 8, 1)
            yield tile - max(tile // 8, 1)
    while True:
        yield tile


def _staged_wants(n_bytes, block, tile_mib):
    n_blocks = n_bytes // block
    chunk = max(((tile_mib << 20) // 4) // block, 1)
    tile = min(4 * chunk, n_blocks)
    chunk = min(chunk, tile)
    if n_blocks > tile and tile > chunk:
        yield chunk
        yield tile - chunk
    while True:
        yield tile


def _generated_wants(n_bytes, block, tile_mib):
    tile = min(max((tile_mib << 20) // block, 1), n_bytes // block)
    while True:
        yield tile


def test_tile_schedules_of_streamed_sources(pkg, ctx, torch_mod, tmp_path):
    """the tile schedules of the three streaming pipelines, seen through the launch counter: every tile is one cell-sponge
    launch (plus one generator launch for generated bytes), so a commit from pinned memory, pageable memory, a file or the
    fake-data generator launches n_tiles - 1 more kernels than the resident commit of the same bytes, with the same root.
    Fresh contexts with 16 MiB tiles cover both starts of the pinned pipeline, rings of two and three tiles, and the
    automatic start, which uses mode 0 on a context's first commit"""
    import os
    torch = torch_mod
    seed, block, cell = 0x5EED, 65536, 2048
    n_bytes = 4800 * block                                                # 300 MiB
    d = torch.empty(n_bytes, dtype=torch.uint8, device="cuda")
    ctx.fake_cells_dev(seed, 0, n_bytes // cell, cell, d.data_ptr())
    torch.cuda.synchronize()
    pinned = torch.empty(n_bytes, dtype=torch.uint8, pin_memory=True)
    pinned.copy_(d)
    torch.cuda.synchronize()
    pageable = d.cpu().numpy()
    path = str(tmp_path / "slot.dat")
    pageable.tofile(path)
    n_file, n_fake = _tiles(4800, _staged_wants(n_bytes, block, 16)), _tiles(4800, _generated_wants(n_bytes, block, 16))
    for ramp, stage_tiles in ((0, 2), (0, 3), (1, 2), (1, 3), (None, None)):
        env = {"CODEX_COMMIT_TILE_MIB": "16", "CODEX_COMMIT_RAMP": ramp, "CODEX_COMMIT_STAGE_TILES": stage_tiles}
        saved = {k: os.environ.pop(k, None) for k in env}
        os.environ.update({k: str(v) for k, v in env.items() if v is not None})
        try:
            c = pkg.Context(0)
        finally:
            for k, v in saved.items():
                os.environ.pop(k, None)
                if v is not None:
                    os.environ[k] = v

        def delta(commit):
            before = c.launches
            with commit() as s:
                return c.launches - before, s.root

        n_pinned = _tiles(4800, _pinned_wants(n_bytes, block, 16, gradual=ramp == 1))   # automatic start: mode 0 at first
        got = [delta(lambda: c.slot_commit_host(pinned.data_ptr(), n_bytes=n_bytes)),
               delta(lambda: c.slot_commit_host(pageable)),
               delta(lambda: c.slot_commit_file(path, n_bytes)),
               delta(lambda: c.slot_commit_fake(seed, n_bytes // cell))]
        resident, root = delta(lambda: c.slot_commit_dev(d.data_ptr(), n_bytes))
        want = [resident + n_pinned - 1, resident + n_file - 1, resident + n_file - 1, resident + 2 * n_fake - 1]
        assert [g[0] for g in got] == want, (ramp, stage_tiles)
        assert all(g[1] == root for g in got), (ramp, stage_tiles)
        c.close()


def test_guard_bands_around_caller_buffers(ctx, torch_mod):
    """device-side memory safety without compute-sanitizer (closed on this pool): every entry point that writes into a
    caller's device buffer is run with ragged sizes (partial warps, partial CTAs, sizes around the launch-width switches)
    between two guard bands, which must come back untouched"""
    torch = torch_mod
    G = 4096

    def guarded(n_bytes):
        buf = torch.full((n_bytes + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
        return buf, buf.data_ptr() + G

    def intact(buf, n_bytes):
        torch.cuda.synchronize()
        return bool((buf[:G] == 0xA5).all()) and bool((buf[G + n_bytes:] == 0xA5).all())

    for cell in (2048, 64, 100):                                         # TMA kernel (two geometries) and the plain-load kernel
        for n_cells in (1, 31, 33, 255, 257, 4735, 4737, 9473, 20001):
            src = synthetic(ctx, torch, (n_cells * cell + 7) // 8 * 8, seed=n_cells)
            out, p = guarded(32 * n_cells)
            ctx.hash_cells_dev(src.data_ptr(), n_cells, cell, p)
            assert intact(out, 32 * n_cells), (cell, n_cells)
    for n in (1, 33, 1000, 37889):
        src = synthetic(ctx, torch, 96 * n, seed=n)
        out, p = guarded(96 * n)
        ctx.permutation_batch_dev(src.data_ptr(), p, n)
        assert intact(out, 96 * n), n
    for n_cells, cell in ((1, 2048), (37, 2048), (300, 64), (129, 100)):
        out, p = guarded(n_cells * cell)
        ctx.fake_cells_dev(99, 5, n_cells, cell, p)
        assert intact(out, n_cells * cell), (n_cells, cell)
    for n_bytes in (8, 4096 + 8, 1 << 20):
        out, p = guarded(n_bytes)
        ctx.fill_synthetic_dev(3, 17, n_bytes, p)
        assert intact(out, n_bytes), n_bytes
    d = synthetic(ctx, torch, 100 * 65536)
    with ctx.slot_commit_range_dev(d.data_ptr(), 100 * 65536, 2048, 65536, 0, 100, 2) as sh:      # 25 level-2 nodes
        _, cnt, _ = sh.subtree_roots()
        out, p = guarded(32 * cnt)
        sh.subtree_roots_copy_dev(p)
        assert cnt == 25 and intact(out, 32 * cnt)


def test_library_allocations_between_guard_bands():
    """CODEX_COMMIT_GUARD=1 puts 4 KiB guard bands around EVERY device allocation the library makes (tree layers, top
    trees, staging tiles, scoped buffers) and aborts the process if a band is damaged when the allocation is freed: a
    representative part of the GPU suite -- ragged slots, every cell path, batches, datasets with all source kinds, the
    sharded entry points, export/import, the geometry fuzz -- must pass unchanged in that mode"""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    select = ("config1_slot or ragged_block_counts or other_cell_and_block_sizes or every_cell_path or export_import or prove_batch_many "
              "or batched_small_slots or dataset_commit_small or dataset_commit_mixed or sharded_entry_points or sharded_commit_equals "
              "or fuzz_geometries or commit_file_vs_oracle or launch_boundary or across_batch_boundaries or segmented_pass_many_trees "
              "or one_cell_slots or batch_fake_300 or synthetic_members_behind or synthetic_tiles_starting or no_byte_unwritten")
    env = dict(os.environ, CODEX_COMMIT_GUARD="1")
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests"), "-m", "gpu", "-x", "-q", "-k", select],
                         capture_output=True, text=True, env=env, timeout=1500, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "CODEX_COMMIT_GUARD" not in res.stderr
    assert " passed" in res.stdout
    # and the mechanism itself: a deliberate one-byte overrun must abort the process in guard mode, and only then
    probe = ("import importlib, sys; sys.path.insert(0, %r); p = importlib.import_module('codex-storage-proofs-circuits_b200'); "
             "c = p.Context(0); print('rc', c.lib.cdx_debug_guard_selftest(c.h))" % ROOT)
    bad = subprocess.run([sys.executable, "-c", probe], capture_output=True, text=True, env=env, timeout=300)
    assert bad.returncode != 0 and "PAST its end" in bad.stderr, bad.stdout + bad.stderr
    off = subprocess.run([sys.executable, "-c", probe], capture_output=True, text=True, env=dict(os.environ, CODEX_COMMIT_GUARD="0"), timeout=300)
    assert off.returncode == 0 and "rc -7" in off.stdout, off.stdout + off.stderr
