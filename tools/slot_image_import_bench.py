#!/usr/bin/env python3
"""What cdx_slot_import costs, and how much of it is the payload check (k_check_image); not part of bench.py.

Commits a synthetic slot (8 GiB by default, 2 KiB cells, 64 KiB blocks), exports its full image (block forest + slot tree,
256 MiB at 8 GiB) and, after cdx_slot_compact, its compact image (slot tree only, 8 MiB).  Each image is imported R times
from pageable host memory; an import ends in a stream synchronise, so the host clock around it is the call's time.  A
separate run under torch.profiler gives the device time of the check kernel and of the host-to-device copies per import;
"without the check" is the import's time minus the check kernel's.  Every import must give the committed root.
Writes one JSON object to the output path.
usage: slot_image_import_bench.py [output = profiles/r3_slot_image_import_8GiB.json] [slot GiB = 8] [R = 10]
"""
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

pkg = importlib.import_module("codex-storage-proofs-circuits_b200")
out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_slot_image_import_8GiB.json")
gib = float(sys.argv[2]) if len(sys.argv) > 2 else 8.0
REPS = int(sys.argv[3]) if len(sys.argv) > 3 else 10
SEED, CELL, BLOCK = 0x1A6E, 2048, 65536
n = int(gib * (1 << 30)) // BLOCK * BLOCK


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=60).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:                      # noqa: BLE001 -- the numbers stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def time_imports(ctx, image, root):
    with ctx.slot_import(image) as s:           # warm-up: module load, pool growth
        assert s.root == root
    ms = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        s = ctx.slot_import(image)
        ms.append((time.perf_counter() - t0) * 1e3)
        assert s.root == root
        s.free()
    return ms


def profiled_device_ms(ctx, image, reps=3):
    """device time per import of the check kernel and of the host-to-device copies, from a profiled run"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.slot_import(image).free()
    check = copy = 0.0
    for e in prof.events():
        dt = getattr(e, "device_time", None)
        if dt is None:
            dt = e.cuda_time
        if "k_check_image" in e.name:
            check += dt
        elif "Memcpy HtoD" in e.name:
            copy += dt
    return check / 1e3 / reps, copy / 1e3 / reps


ctx = pkg.Context(0)
d = torch.empty(n, dtype=torch.uint8, device="cuda")
ctx.fill_synthetic_dev(SEED, 0, n, d.data_ptr())
torch.cuda.synchronize()
slot = ctx.slot_commit_dev(d.data_ptr(), n, CELL, BLOCK)
root = slot.root
n_cells, n_blocks, bd, sd = slot.shape
del d
torch.cuda.empty_cache()
images = {"full": slot.export()}
slot.compact()
images["compact"] = slot.export()
slot.free()

res = {"tool": "tools/slot_image_import_bench.py", **gpu_info(), "slot_bytes": n, "cell": CELL, "block": BLOCK, "n_cells": n_cells,
       "n_blocks": n_blocks, "block_depth": bd, "slot_depth": sd, "reps": REPS, "source": "pageable host memory (Python bytes)"}
for kind, image in images.items():
    ms = time_imports(ctx, image, root)
    check_ms, copy_ms = profiled_device_ms(ctx, image)
    nodes = (len(image) - 56) // 32
    compressions = nodes - (n_cells if kind == "full" else n_blocks)      # every stored node above the bottom level
    med = statistics.median(ms)
    res[kind] = {"image_bytes": len(image), "stored_nodes": nodes, "compressions_checked": compressions,
                 "import_ms_median": round(med, 3), "import_ms_min": round(min(ms), 3), "import_ms_max": round(max(ms), 3),
                 "check_kernel_ms": round(check_ms, 3), "h2d_copy_ms": round(copy_ms, 3),
                 "import_without_check_ms": round(med - check_ms, 3), "check_share": round(check_ms / med, 4)}
ctx.close()
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    json.dump(res, f, indent=1)
    f.write("\n")
print(json.dumps(res))
