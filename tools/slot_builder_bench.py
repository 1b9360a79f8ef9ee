#!/usr/bin/env python3
"""What a slot builder (cdx_slot_builder_*) costs against cdx_slot_commit_host on the same bytes; not part of bench.py.

An 8 GiB slot (2 KiB cells, 64 KiB blocks) of seeded random bytes in pageable host memory (a numpy array, far larger than
the 126 MB L2).  Cases, each timed R >= 5 times on the host clock around calls that end synchronised (median reported):
  1. cdx_slot_commit_host on the whole slot;
  2. a builder fed with one add of the whole slot;
  3. 64 KiB adds (one block each) in block order;
  4. 64 KiB adds in a seeded random order;
  5. 1 MiB adds (16 blocks) in a seeded random order.
Cases 2-5 run with keep_forest 1 (full handle) and 0 (compact handle); a builder's time runs from create to the end of
finish.  Every root must equal case 1's.  Also reported: each handle's cdx_slot_device_bytes and the builder's staging
memory, computed from its tile sizes (four pinned chunks of a quarter tile, two id tables; two device tiles, two id tables
and two scratch forests).  Writes one JSON object to the output path.
usage: slot_builder_bench.py [output = profiles/r3_slot_builder_8GiB.json] [slot GiB = 8] [R = 5]
"""
import importlib
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

pkg = importlib.import_module("codex-storage-proofs-circuits_b200")
out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_slot_builder_8GiB.json")
gib = float(sys.argv[2]) if len(sys.argv) > 2 else 8.0
REPS = max(5, int(sys.argv[3]) if len(sys.argv) > 3 else 5)
SEED, CELL, BLOCK, TILE_MIB = 0x5B1D, 2048, 65536, 256
n = int(gib * (1 << 30)) // BLOCK * BLOCK
n_blocks = n // BLOCK


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=60).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:                      # noqa: BLE001 -- the numbers stand without it, but say so
        return {"gpu": "unknown", "power_limit": f"unknown ({e})"}


def staging_bytes(n_blocks, cell, block, tile_mib):
    """the builder's own memory, from the tile sizes of cdx_slot_builder_create"""
    tile = max(1, min(n_blocks, (tile_mib << 20) // block))
    chunk = -(-tile // 4)
    cpb = block // cell
    cells = tile * cpb
    bd = 1 if cpb == 1 else cpb.bit_length() - 1
    forest = sum(cells if cpb == 1 else cells >> lvl for lvl in range(bd + 1))
    return {"tile_blocks": tile, "chunk_blocks": chunk, "pinned_host_bytes": -(-tile // chunk) * chunk * block + 2 * 8 * tile,
            "device_bytes": 2 * (tile * block + 8 * tile + 32 * forest)}


data = np.random.default_rng(SEED).integers(0, 1 << 64, n // 8, dtype=np.uint64).view(np.uint8)
base = data.ctypes.data
ctx = pkg.Context(0)


def commit_host():
    s = ctx.slot_commit_host(data, CELL, BLOCK)
    return s


def builder(keep, adds):
    def run():
        b = ctx.slot_builder(n_blocks, CELL, BLOCK, keep_forest=keep)
        for first, k in adds:
            b.add(first, base + first * BLOCK, k * BLOCK)
        s = b.finish()
        b.free()
        return s
    return run


rnd = random.Random(SEED)
in_order = [(j, 1) for j in range(n_blocks)]
shuffled = rnd.sample(in_order, n_blocks)
mib_runs = [(j, min(16, n_blocks - j)) for j in range(0, n_blocks, 16)]
rnd.shuffle(mib_runs)
cases = [("1_commit_host", None, commit_host)]
for keep in (1, 0):
    cases += [(f"2_builder_one_add_keep{keep}", keep, builder(keep, [(0, n_blocks)])),
              (f"3_builder_64KiB_in_order_keep{keep}", keep, builder(keep, in_order)),
              (f"4_builder_64KiB_random_keep{keep}", keep, builder(keep, shuffled)),
              (f"5_builder_1MiB_random_keep{keep}", keep, builder(keep, mib_runs))]

res = {"tool": "tools/slot_builder_bench.py", **gpu_info(), "slot_bytes": n, "cell": CELL, "block": BLOCK, "n_blocks": n_blocks,
       "tile_mib": TILE_MIB, "reps": REPS, "source": "pageable host memory (numpy array of seeded random bytes)",
       "builder_staging": staging_bytes(n_blocks, CELL, BLOCK, TILE_MIB), "cases": {}}
root = None
for name, keep, run in cases:
    s = run()                                  # warm-up: module load, pool growth, pinned allocations
    if root is None:
        root = s.root
    assert s.root == root, name
    dev_bytes = s.device_bytes
    s.free()
    secs = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        s = run()
        secs.append(time.perf_counter() - t0)
        assert s.root == root, name
        s.free()
    med = statistics.median(secs)
    res["cases"][name] = {"keep_forest": keep, "s_median": round(med, 4), "s_min": round(min(secs), 4), "s_max": round(max(secs), 4),
                          "gbs_median": round(n / med / 1e9, 3), "handle_device_bytes": dev_bytes}
    print(name, res["cases"][name], flush=True)
res["root_hex"] = hex(root)
ctx.close()
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    json.dump(res, f, indent=1)
    f.write("\n")
print(json.dumps(res))
