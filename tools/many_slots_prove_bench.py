#!/usr/bin/env python3
"""Challenges against many compact slots: M calls of cdx_slot_prove_from_source (one per slot) against one call of
cdx_slots_prove_from_source for all of them; not part of bench.py.

Commits power-of-two synthetic slots on the device and compacts each one: 256 slots of 256 MiB and a few slots of 1 GiB,
whose slot trees are two levels deeper.  For M = 1, 16 and 256 of the 256 MiB slots, and for all 256 with the 1 GiB slots
beside them, with S samples per challenge and K = 1 and 10 challenges per slot, it times the loop of one-slot calls and
the one many-slot call.  Every answer of the many-slot call must equal the slot's own answer byte for byte and
reconstruct that slot's root in two stages (cdx_reconstruct_roots_host).  Prints one JSON line.
usage: many_slots_prove_bench.py [S = 100] [number of 1 GiB slots = 4]
"""
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

pkg = importlib.import_module("codex-storage-proofs-circuits_b200")
capi = pkg.capi
S = int(sys.argv[1]) if len(sys.argv) > 1 else 100
N_BIG = int(sys.argv[2]) if len(sys.argv) > 2 else 4
DEPTH, CELL, BLOCK = 32, 2048, 65536
SMALL, BIG, N_SMALL = 256 << 20, 1 << 30, 256
KS = (1, 10)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=60).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:                      # noqa: BLE001 -- the numbers stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


ctx = pkg.Context(0)
lib, chk = ctx.lib, ctx._chk
# slot m: synthetic bytes with seed 1000 + m, committed from the device, then compacted
sizes = [SMALL] * N_SMALL + [BIG] * N_BIG
d = torch.empty(BIG, dtype=torch.uint8, device="cuda")
slots, descs = [], []
for m, n in enumerate(sizes):
    seed = 1000 + m
    ctx.fill_synthetic_dev(seed, 0, n, d.data_ptr())
    torch.cuda.synchronize()
    slot = ctx.slot_commit_dev(d.data_ptr(), n, CELL, BLOCK)
    slot.compact()
    torch.cuda.synchronize()
    slots.append(slot)
    descs.append((capi.SRC_SYNTHETIC, seed, n))
del d
torch.cuda.empty_cache()
shapes = [s.shape for s in slots]
roots = [capi.f2b(s.root) for s in slots]


def entropy(m, j):
    return capi.f2b((0x9e3779b97f4a7c15 * (m + 1) + 0x632be59bd9b4e019 * (j + 1)) % (1 << 250))


def buffers(rows):
    total = rows * S
    return ((C.c_uint64 * total)(), C.create_string_buffer(32 * total * DEPTH), C.create_string_buffer(32 * total), C.create_string_buffer(CELL * total))


def verify(m, idx, paths, leaves, first, count):
    """samples [first, first + count) answer slot m: two-stage reconstruction of its root"""
    n_cells, n_blocks, bd, sd = shapes[m]
    cpb = n_cells // n_blocks
    ii = idx[first:first + count]
    in_block = (C.c_uint64 * count)(*[i % cpb for i in ii])
    in_slot = (C.c_uint64 * count)(*[i // cpb for i in ii])
    blk, top = C.create_string_buffer(32 * count), C.create_string_buffer(32 * count)
    p0 = C.addressof(paths) + 32 * DEPTH * first
    chk(lib.cdx_reconstruct_roots_host(ctx.h, C.addressof(leaves) + 32 * first, C.addressof(in_block), cpb, p0, DEPTH, bd, count, C.addressof(blk)))
    chk(lib.cdx_reconstruct_roots_host(ctx.h, C.addressof(blk), C.addressof(in_slot), n_blocks, p0 + 32 * bd, DEPTH, sd, count, C.addressof(top)))
    assert top.raw == roots[m] * count, f"an answer does not reconstruct the root of slot {m}"


def timed(fn, reps=3):
    ts = []
    for _ in range(reps + 1):                   # the first call is the warm-up
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts[1:]), ts[1:]


configs = [("256MiBx1", [0]), ("256MiBx16", list(range(16))), ("256MiBx256", list(range(N_SMALL)))]
if N_BIG:
    configs.append((f"256MiBx256+1GiBx{N_BIG}", list(range(N_SMALL + N_BIG))))
result = {}
for name, ms in configs:
    for K in KS:
        rows = len(ms) * K
        # one call per slot, each with its K challenges, into the same output layout (slot-major rows)
        idx, paths, leaves, cells = buffers(rows)
        per_slot = []
        for r, m in enumerate(ms):
            arr, keep = capi.make_descs([descs[m]])
            ent = b"".join(entropy(m, j) for j in range(K))
            per_slot.append((m, arr, keep, ent, r * K * S))

        def loop():
            for m, arr, _, ent, off in per_slot:
                chk(lib.cdx_slot_prove_from_source(slots[m].h, arr, capi._addr(ent), K, S, DEPTH, C.addressof(idx) + 8 * off,
                                                   C.addressof(paths) + 32 * DEPTH * off, C.addressof(leaves) + 32 * off,
                                                   C.addressof(cells) + CELL * off))
        t_loop, all_loop = timed(loop)
        want = (bytes(idx), paths.raw, leaves.raw, cells.raw)
        # the same rows in one call
        arr, keep = capi.make_descs([descs[m] for m in ms for _ in range(K)])
        handles = (C.c_void_p * rows)(*[slots[m].h for m in ms for _ in range(K)])
        ents = b"".join(entropy(m, j) for m in ms for j in range(K))
        idx, paths, leaves, cells = buffers(rows)
        t_one, all_one = timed(lambda: chk(lib.cdx_slots_prove_from_source(handles, arr, capi._addr(ents), rows, S, DEPTH, idx, paths, leaves, cells)))
        assert (bytes(idx), paths.raw, leaves.raw, cells.raw) == want, (name, K)
        for r, m in enumerate(ms):
            verify(m, idx, paths, leaves, r * K * S, K * S)
        cpb = BLOCK // CELL
        unique = len({(r // K, i // cpb) for r in range(rows) for i in idx[r * S:(r + 1) * S]})
        result[f"{name}_K{K}"] = {
            "slots": len(ms), "challenges": rows, "unique_blocks": unique, "rehashed_gb": unique * BLOCK / 1e9,
            "per_slot_calls_ms": 1e3 * t_loop, "per_slot_calls_all_ms": [1e3 * t for t in all_loop],
            "one_call_ms": 1e3 * t_one, "one_call_all_ms": [1e3 * t for t in all_one],
            "speedup": t_loop / t_one, "one_call_rehash_gb_per_s": unique * BLOCK / 1e9 / t_one,
        }
for s in slots:
    s.free()

print(json.dumps({
    **gpu_info(), "samples_per_challenge": S, "slot_sizes": {"256MiB": N_SMALL, "1GiB": N_BIG},
    "slot_depths": sorted({sh[3] for sh in shapes}), "source": "synthetic (generated on the device)", **result,
    "every_answer_equals_the_per_slot_answer_and_reconstructs_its_root": True,
}))
