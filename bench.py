#!/usr/bin/env python3
"""bench.py -- slot-commit throughput on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py --gpus N --steps K --warmup W                (N = 1; N > 1 under torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W   (the CPU path, timed on the host cores)

A "step" is one commitment of the workload: every 2048-byte cell through the Poseidon2 rate-2 sponge, every 64 KiB
block tree, the slot tree, and the 32-byte root read back.  Workload at N = 1: BASELINE.json configs[2], a single
10 GiB synthetic slot (163 840 blocks, not a power of two).  At N > 1 each rank holds 10 GiB of one N x 10 GiB slot
(weak scaling) and commits it through ONE C-ABI call, cdx_slot_commit_sharded_*: its block range on its own GPU, one NCCL
collective inside the library for the level-15 sub-tree roots (5 x 32 B per rank), the replicated top tree.  torch
supplies the process group that broadcasts the library's 128-byte communicator id, the barrier and the device buffers --
nothing on the data path.

Beside the headline the line carries (each outside the headline's timed region, each with its own timing):
  N = 1   small_slots      BASELINE configs[0] (eleven 4 MiB fake-data slots + dataset root) through the batched entry point,
                           and 1000 x 4 MiB slots batched vs one by one
  N > 1   config4_strong   BASELINE configs[3]: ONE 100 GiB slot split over the ranks, root checked against the known value
          sharded_root_check  rank 0 re-commits the whole N x 10 GiB slot alone and compares roots
  N = 8   config5          BASELINE configs[4] at quarter scale: 250 slots (non-power-of-two), 0.25-25 GiB, cdx_dataset_commit

  value     whole-job GB/s with the slot bytes already resident in HBM (CUDA events, max over ranks)
  e2e       the same through the host-buffer C-ABI call (pinned host slot -> cdx_slot_commit[_range]_host), H2D of
            every byte inside the timed region, root read back
  roofline  the dominant kernel (k_hash_cells) timed alone with CUDA events; bound = FMA-heavy-pipe integer multiply
            issue (DESIGN.md "Roofline"), peak = best IMAD.WIDE.U32 rate measured by probe kernels in the same run;
            an `hbm` sub-object shows HBM is three orders of magnitude from binding
  cpu_baseline  oracle (C restatement of the reference path; the Nim toolchain is absent) on a bounded sample

--dump-outputs DIR writes what the last timed step of the headline committed (rank 0's part at N > 1) as float64 .npy
files, each field element as 8 little-endian 32-bit limbs (exact in float64), so that two builds can be compared output
for output: slot_root, block_hashes and cell_hashes, each layer whole up to 2^18 nodes and otherwise a seeded sample of
32-node windows, with the global node numbers beside it (<name>_index.npy).  Under 40 MB whatever the slot size.

Nothing is written into the source tree (it may be read-only): the host-tuned oracle build goes to a temporary directory.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PKG = "codex-storage-proofs-circuits_b200"
CELL, BLOCK = 2048, 65536
PERMS_PER_BLOCK = 32 * 34 + 31              # BASELINE.md section 2
MODMUL_PER_PERM = 240
IMAD_PER_MODMUL = 136                        # 128 IMAD.WIDE.U32 + 8 IMAD (8x32-bit-limb CIOS)
SEED = 0xC0DE


def slot_tree_perms(n_blocks: int) -> int:
    """compressions in the slot tree over n block hashes (merkle/bn254.nim:38-53)"""
    total, n, bottom = 0, n_blocks, True
    while bottom or n > 1:
        total += (n + 1) // 2
        n, bottom = (n + 1) // 2, False
    return total


def total_perms(n_blocks: int) -> int:
    return n_blocks * PERMS_PER_BLOCK + slot_tree_perms(n_blocks)


def layout(args, world: int):
    """(n_total_blocks, top_level, ranges, scaling) -- the same for both arms"""
    sharded = importlib.import_module(PKG + ".sharded")
    if args.total_gib > 0:                             # strong scaling: one slot, 2^T-aligned chunks dealt evenly
        n_total_blocks = int(args.total_gib * (1 << 30)) // BLOCK
        top_level, ranges = sharded.plan_block_ranges(n_total_blocks, world)
        return n_total_blocks, top_level, ranges, "strong"
    blocks_per_gpu = int(args.slot_gib * (1 << 30)) // BLOCK   # weak scaling: every rank holds --slot-gib of one N x larger slot
    top_level, ranges = sharded.fixed_ranges(blocks_per_gpu, world)
    return blocks_per_gpu * world, top_level, ranges, "weak"


def make_config(args, world: int, n_total_blocks: int, top_level: int, ranges) -> dict:
    per_gpu = max(c for _, c in ranges) * BLOCK
    return {"workload": (f"single {args.total_gib:g} GiB synthetic slot split over {world} GPU(s)" if args.total_gib > 0 else
                         f"single {args.slot_gib:g} GiB-per-GPU synthetic slot") +
                        f" ({n_total_blocks} blocks of 64 KiB, 2048-byte cells): cell sponge + block trees + slot tree + root",
            "bytes_per_step": n_total_blocks * BLOCK, "cell_size": CELL, "block_size": BLOCK, "seed": SEED,
            "parallelism": "1 GPU" if world == 1 else f"{world} ranks x block-range shards, level-{top_level} roots combined by one NCCL collective "
                                                       "inside cdx_slot_commit_sharded_*",
            "l2": f"inputs ({per_gpu / 2**30:.1f} GiB per GPU) are larger than L2; no flush needed"}


# ---------------------------------------------------------------------------------------------------------------
# synthetic bytes on the host (numpy twin of k_fill_synthetic) for the CPU legs

def synthetic_bytes_host(seed: int, first_word: int, n_bytes: int):
    import numpy as np
    with np.errstate(over="ignore"):
        i = np.arange(n_bytes // 8, dtype=np.uint64)
        z = i + np.uint64((seed + first_word + 0x9e3779b97f4a7c15) & (2**64 - 1))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
        z = z ^ (z >> np.uint64(31))
    return z.view(np.uint8)


# ---------------------------------------------------------------------------------------------------------------
# --dump-outputs

DUMP_MAX_NODES = 1 << 18                     # per layer: 2^18 nodes x 8 limbs x 8 bytes = 16 MiB (+ 2 MiB of node numbers)
DUMP_WINDOW = 32                             # sampled layers are read in windows of 32 nodes (one block's cells)


def dump_layer(slot, tree: int, level: int, first: int, count: int, rng):
    """(node numbers, (n, 8) float64 limbs) of nodes [first, first + count) of one retained layer: all of them up to
    DUMP_MAX_NODES, else a seeded sample of DUMP_WINDOW-node windows"""
    import numpy as np
    if count <= DUMP_MAX_NODES:
        windows = [(first, count)]
    else:
        starts = np.sort(rng.choice(count // DUMP_WINDOW, DUMP_MAX_NODES // DUMP_WINDOW, replace=False))
        windows = [(first + int(s) * DUMP_WINDOW, DUMP_WINDOW) for s in starts]
    idx = np.concatenate([np.arange(f, f + n, dtype=np.float64) for f, n in windows])
    raw = b"".join(int(v).to_bytes(32, "little") for f, n in windows for v in slot.read_layer(tree, level, f, n))
    return idx, np.frombuffer(raw, dtype="<u4").reshape(-1, 8).astype(np.float64)


def dump_outputs(out_dir: str, slot, first_block: int, n_blocks: int) -> None:
    """the slot's root, its block hashes and its cell hashes (of blocks [first_block, first_block + n_blocks)) as .npy"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(SEED)
    cells_per_block = BLOCK // CELL
    out = {"slot_root": np.frombuffer(slot.root.to_bytes(32, "little"), dtype="<u4").reshape(1, 8).astype(np.float64)}
    out["block_hashes_index"], out["block_hashes"] = dump_layer(slot, 1, 0, first_block, n_blocks, rng)
    out["cell_hashes_index"], out["cell_hashes"] = dump_layer(slot, 0, 0, first_block * cells_per_block, n_blocks * cells_per_block, rng)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    print(f"dumped {', '.join(out)} ({sum(a.nbytes for a in out.values()) / 2**20:.1f} MiB) to {out_dir}", file=sys.stderr)


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def tune_oracle(threads: int):
    """The CPU legs should not be handicapped by a slow build: compile the oracle for THIS host (-O3 -march=native) and
    keep the faster of its two S-box forms (dedicated squaring / general product for x^2 and x^4).  Returns
    (description, seconds for a 64 MiB commitment)."""
    from oracle import coracle
    native = coracle.use_native()
    best = None
    for use_sqr in (True, False):
        coracle.set_use_sqr(use_sqr)
        dt, _ = time_oracle_commit(64 << 20, threads)
        if best is None or dt < best[1]:
            best = (use_sqr, dt)
    coracle.set_use_sqr(best[0])
    desc = ("gcc -O3 -march=native on this host" if native else "portable -O3 -mbmi2 -madx build") + \
           (", dedicated 10-product squaring" if best[0] else ", general CIOS product for the squarings (faster here than the dedicated squaring)")
    return desc, best[1]


def time_oracle_commit(sample_bytes: int, threads: int, reps: int = 1):
    """seconds per commitment of `sample_bytes` of the synthetic slot on the host cores (oracle = checker, timed here
    only as the reported CPU baseline)"""
    from oracle import coracle
    coracle.build()
    buf = synthetic_bytes_host(SEED, 0, sample_bytes)
    best = None
    root = None
    for _ in range(reps):
        t0 = time.perf_counter()
        root, _, _ = coracle.commit_slot((buf.ctypes.data, sample_bytes), CELL, BLOCK, n_threads=threads)
        dt = time.perf_counter() - t0
        best = dt if best is None or dt < best else best
    return best, root


# ---------------------------------------------------------------------------------------------------------------
# clocks during the timed region (B200_PROFILING.md recipe)

class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_id: str):
        self.gpu_id, self.rows, self.proc, self.thread = gpu_id, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.gpu_id, "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------

def run_reference(args) -> None:
    """The reference arm: the path's CPU implementation on the box's host cores.  The Nim reference cannot be built
    here (no nim/nimble; constantine and nim-poseidon2 are un-vendored), so this is the oracle port, all threads, compiled
    on this machine with -O3 -march=native (dedicated squaring, MULX/ADX through unsigned __int128)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    # one step = one commitment of a bounded prefix of the workload's synthetic slot; 1 GiB unless the whole run would
    # exceed ~3 minutes on this host, in which case the prefix shrinks (never below 256 MiB) -- the real size is reported
    build_desc, probe_s = tune_oracle(threads)
    rate = (64 << 20) / probe_s
    budget_s = 180.0
    sample = args.ref_sample_mib << 20
    while sample > (256 << 20) and sample * (args.steps + 1) / rate > budget_s:
        sample //= 2
    time_oracle_commit(sample, threads)                      # one untimed pass (touches the pages); a CPU needs no more warm-up
    t = 0.0
    for _ in range(args.steps):
        dt, _ = time_oracle_commit(sample, threads)
        t += dt
    gbs = sample * args.steps / t / 1e9
    n_total_blocks, top_level, ranges, scaling = layout(args, args.gpus)
    cfg = make_config(args, args.gpus, n_total_blocks, top_level, ranges)
    cfg["reference_sample"] = (f"each reference step commits the first {sample >> 20} MiB ({sample // BLOCK} blocks) of that slot on "
                               f"{threads} host threads, not the whole slot: a rate, scaled to the same unit")
    cfg["reference_sample_bytes"] = sample
    line = {
        "impl": "reference", "metric": "slot commit GB/s (with Poseidon2 perms/s)", "value": gbs, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "u64x4 (BN254 Fr, Montgomery)", "data": "synthetic",
        "config": cfg,
        "perms_per_s": total_perms(sample // BLOCK) * args.steps / t,
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "port",
                         "sample": f"first {sample >> 20} MiB of the workload's synthetic slot per step, {threads} threads over blocks; "
                                   "C restatement of reference/nim/proof_input (Nim toolchain absent), " + build_desc},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--slot-gib", type=float, default=10.0, help="GiB of slot data per GPU (default: BASELINE config 3, 10 GiB)")
    ap.add_argument("--total-gib", type=float, default=0.0,
                    help="strong scaling: ONE slot of this many GiB split over the ranks by plan_block_ranges (BASELINE config 4: 100); "
                         "overrides --slot-gib")
    ap.add_argument("--ref-sample-mib", type=int, default=1024, help="bytes per step of the --impl reference CPU run (shrinks on slow hosts)")
    ap.add_argument("--cpu-sample-mib", type=int, default=1024, help="sample committed once for cpu_baseline (N=1, rank 0)")
    ap.add_argument("--no-extras", action="store_true", help="skip small_slots / config4_strong / sharded_root_check / config5")
    ap.add_argument("--config5", default="auto", choices=["auto", "on", "off"], help="dataset commit (BASELINE configs[4]); auto = only at 8 GPUs")
    ap.add_argument("--config5-scale", type=float, default=0.25, help="slot sizes are 1-100 GiB times this factor")
    ap.add_argument("--config5-slots", type=int, default=250)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as .npy files under DIR")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    sys.dont_write_bytecode = True              # nothing is written into the tree, not even __pycache__
    if args.impl == "reference":
        return run_reference(args)

    # only the JSON line may reach stdout: library chatter (e.g. "NCCL version ..." printed at communicator creation)
    # is sent to stderr for the duration of the run
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    build_mod = importlib.import_module(PKG + ".build")
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        build_mod.ensure_built()                                 # no-op when the in-tree build exists
    else:
        t_wait = time.time()
        while not os.path.exists(build_mod.LIB) and time.time() - t_wait < 600:
            time.sleep(1.0)
    pkg = importlib.import_module(PKG)
    sharded = importlib.import_module(PKG + ".sharded")

    rank, world, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = pkg.Context(local_rank)                      # raises if libcodexcommit.so or the GPU is missing: no fallback
    stream = torch.cuda.ExternalStream(ctx.stream)     # the library's compute stream, so events see its kernels
    comm = sharded.comm_from_torch(ctx) if world > 1 else None    # the library's own NCCL communicator (cdx_comm_init_rank)

    n_total_blocks, top_level, ranges, scaling = layout(args, world)
    first_block, my_blocks = ranges[rank]
    n_bytes = my_blocks * BLOCK

    d_slot = torch.empty(n_bytes, dtype=torch.uint8, device="cuda")
    ctx.fill_synthetic_dev(SEED, first_block * (BLOCK // 8), n_bytes, d_slot.data_ptr())
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    kept = []                                         # --dump-outputs: the latest step's slot, read after the timed region

    def commit_resident():
        if world == 1:
            slot = ctx.slot_commit_dev(d_slot.data_ptr(), n_bytes, CELL, BLOCK)
        else:
            slot = ctx.slot_commit_sharded_dev(comm, d_slot.data_ptr(), n_bytes, CELL, BLOCK, first_block, n_total_blocks, top_level)
        root = slot.root                              # 32-byte D2H, synchronises the stream
        if args.dump_outputs:                         # free the previous step's slot instead: still one free per step
            for s in kept:
                s.free()
            kept[:] = [slot]
        else:
            slot.free()
        return root

    def timed(fn, steps):
        """CUDA events on the library stream + wall clock, both bracketed by barrier + synchronize; max over ranks"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        out = None
        for _ in range(steps):
            out = fn()
        e1.record(stream)
        e1.synchronize()
        barrier()
        wall = time.perf_counter() - t0
        ev = e0.elapsed_time(e1) / 1e3
        t = torch.tensor([ev, wall], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), out

    gpu_id = str(local_rank)
    try:
        gpu_id = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        pass

    # ---- resident-data run (value) ----
    for _ in range(args.warmup):
        root = commit_resident()
    sampler = ClockSampler(gpu_id)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launches
    ev_s, wall_s, root = timed(commit_resident, args.steps)
    launches = ctx.launches - launches0
    clocks = sampler.stop() if rank == 0 else None
    total_bytes = n_total_blocks * BLOCK
    value = total_bytes * args.steps / ev_s / 1e9
    perms_step = total_perms(n_total_blocks)
    if kept:
        if rank == 0:
            dump_outputs(args.dump_outputs, kept[0], first_block, my_blocks)
        kept.pop().free()

    # ---- dominant kernel alone (roofline) ----
    n_cells = n_bytes // CELL
    d_hashes = torch.empty(n_cells * 32, dtype=torch.uint8, device="cuda")
    ctx.hash_cells_dev(d_slot.data_ptr(), n_cells, CELL, d_hashes.data_ptr())
    k_ev, _, _ = timed(lambda: ctx.hash_cells_dev(d_slot.data_ptr(), n_cells, CELL, d_hashes.data_ptr()), args.steps)
    k_ms = 1e3 * k_ev / args.steps
    del d_hashes
    imad_wide_rz, _ = ctx.probe_imad_rate(0)        # IMAD.WIDE.U32 Rd,Ra,Rb,RZ (no carry), product fed back into the multiplicand
    imad_wide_x, _ = ctx.probe_imad_rate(1)         # IMAD.WIDE.U32.X carry chains, the form the Montgomery rows use
    imad32, _ = ctx.probe_imad_rate(2)              # 32-bit IMAD, for context: twice the rate of any 32x32->64 form
    imad_wide = max(imad_wide_rz, imad_wide_x)
    kernel_imads = n_cells * 34 * MODMUL_PER_PERM * IMAD_PER_MODMUL
    achieved = kernel_imads / (k_ms * 1e-3)
    hbm_peak = None
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        hbm_src = "measured (MEASURED_PEAKS.json)"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    alg_bytes = n_cells * (CELL + 32)
    roofline = {
        "kernel": "k_hash_cells_tma", "bound": "imad",
        "bound_note": "FMA-heavy pipe: IMAD.WIDE.U32 issue rate; neither hbm nor tensor (see the hbm sub-object and DESIGN.md section 4)",
        "achieved": achieved / 1e12, "peak": imad_wide / 1e12, "unit": "T int-multiply instr/s", "frac": achieved / imad_wide,
        "peak_source": "best IMAD.WIDE.U32 rate measured in this run by cdx_probe_imad_rate (max of the no-carry and the carry-chain form); "
                       "MEASURED_PEAKS.json has no integer peak",
        "note": "achieved = 136 multiply instructions (schoolbook 8x32-bit CIOS) x 240 modmuls x 34 perms x cells / kernel time; the kernel "
                "executes fewer (dedicated 36-product squaring), so frac can exceed 1 -- SURVEY.md 8d: no credit in the denominator",
        "probe_rates_T_per_s": {"imad_wide_u32_no_carry": imad_wide_rz / 1e12, "imad_wide_u32_x_carry_chain": imad_wide_x / 1e12, "imad_u32": imad32 / 1e12},
        "kernel_ms": k_ms, "algorithmic_imads_per_launch": kernel_imads, "modmuls_per_s": achieved / IMAD_PER_MODMUL,
        "traffic": None,
        "hbm": {"achieved": alg_bytes / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": alg_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak,
                "peak_source": hbm_src, "algorithmic_bytes_per_launch": alg_bytes},
    }
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")    # dram bytes from the committed `ncu --set full` capture
    if os.path.exists(traffic_file):
        try:
            tj = json.load(open(traffic_file))
            roofline["traffic"] = tj["dram_bytes_per_slot_byte"] * n_bytes
            roofline["traffic_note"] = ("dram__bytes_read.sum + dram__bytes_write.sum of k_hash_cells_tma, scaled per slot byte from the "
                                        f"{tj['slot_bytes_in_launch'] >> 30} GiB launch captured in {tj['source']}")
        except Exception:
            pass

    # ---- BASELINE config 2: 2^20 independent permutations (kernel time, best of 10) ----
    n_perm = 1 << 20
    d_pin = torch.empty(96 * n_perm, dtype=torch.uint8, device="cuda")
    d_pout = torch.empty_like(d_pin)
    ctx.fill_synthetic_dev(1, 0, 96 * n_perm, d_pin.data_ptr())
    ctx.permutation_batch_dev(d_pin.data_ptr(), d_pout.data_ptr(), n_perm)
    best_perm = None
    for _ in range(10):
        p_ev, _, _ = timed(lambda: ctx.permutation_batch_dev(d_pin.data_ptr(), d_pout.data_ptr(), n_perm), 1)
        best_perm = p_ev if best_perm is None or p_ev < best_perm else best_perm
    perm_batch = {"n": n_perm, "ms": 1e3 * best_perm, "perms_per_s": n_perm / best_perm,
                  "note": "k_permutation_batch incl. to/from Montgomery form (6 extra modmuls per permutation), per GPU"}
    del d_pin, d_pout

    # ---- end to end through the host-buffer ABI ----
    e2e = None
    if not args.no_e2e:
        h_slot = torch.empty(n_bytes, dtype=torch.uint8, pin_memory=True)
        h_slot.copy_(d_slot)
        torch.cuda.synchronize()
        h_np = h_slot.numpy()

        def commit_host():
            if world == 1:
                slot = ctx.slot_commit_host(h_np, CELL, BLOCK)
                r = slot.root
                slot.free()
                return r
            sh = ctx.slot_commit_sharded_host(comm, h_np, n_bytes, CELL, BLOCK, first_block, n_total_blocks, top_level)
            r = sh.root
            sh.free()
            return r

        for _ in range(min(args.warmup, 2)):
            r2 = commit_host()
        _, e2e_wall, r2 = timed(commit_host, args.steps)
        assert r2 == root, "host-buffer path and resident path disagree on the slot root"
        e2e = {"value": total_bytes * args.steps / e2e_wall / 1e9, "unit": "GB/s", "h2d_bytes_per_step": total_bytes, "d2h_bytes_per_step": 32 * world,
               "ms_per_step": 1e3 * e2e_wall / args.steps,
               "api": "cdx_slot_commit_host + cdx_slot_root" if world == 1 else
                      "cdx_slot_commit_sharded_host + cdx_slot_root (NCCL inside libcodexcommit.so; communicator from cdx_comm_init_rank)",
               "timing": "wall clock bracketed by barrier + cudaDeviceSynchronize, max over ranks"}
        del h_slot

    # ---- CPU baseline beside it (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = host_threads()
        sample = min(args.cpu_sample_mib << 20, n_bytes)
        build_desc, probe_s = tune_oracle(threads)            # -O3 -march=native compiled on this host, faster S-box form
        while sample > (256 << 20) and sample / ((64 << 20) / probe_s) > 30.0:     # keep the leg near 10-30 s on slow hosts
            sample //= 2
        dt, cpu_root = time_oracle_commit(sample, threads)
        # the sample doubles as a parity check at bench size: GPU root of the same prefix must equal the oracle's
        with ctx.slot_commit_dev(d_slot.data_ptr(), sample, CELL, BLOCK) as s:
            assert s.root == cpu_root, "GPU and oracle disagree on the sample root"
        cpu = {"value": sample / dt / 1e9, "unit": "GB/s", "cores": threads, "kind": "port",
               "perms_per_s": total_perms(sample // BLOCK) / dt,
               "sample": f"first {sample >> 20} MiB of the same synthetic slot, one commitment, {threads} threads over blocks "
                         "(C restatement of reference/nim/proof_input; Nim toolchain absent; " + build_desc + "); root checked equal to the GPU's"}

    # ---- the other BASELINE configs, each with its own timing, outside the headline's timed region ----
    extras = {}
    del d_slot
    torch.cuda.empty_cache()
    if not args.no_extras:
        extras = run_extras(args, torch, dist, pkg, ctx, comm, stream, rank, world, value, timed, barrier)

    if rank == 0:
        line = {
            "metric": "slot commit GB/s (with Poseidon2 perms/s)", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * ev_s / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "u32x8 (BN254 Fr, 256-bit Montgomery integers)", "data": "synthetic",
            "config": make_config(args, world, n_total_blocks, top_level, ranges),
            "perms_per_s": perms_step * args.steps / ev_s, "perms_per_step": perms_step,
            "slot_root": hex(root), "wall_ms_per_step": 1e3 * wall_s / args.steps,
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu,
            "perm_batch_2^20": perm_batch,
        }
        line.update(extras)
        if "sharded_root_check" in extras:
            extras["sharded_root_check"]["equals_sharded_root"] = extras["sharded_root_check"]["whole_slot_root_one_gpu"] == hex(root)
            assert extras["sharded_root_check"]["equals_sharded_root"], "sharded and whole-slot roots differ"
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if comm is not None:
        comm.destroy()
    if world > 1:
        dist.destroy_process_group()


KNOWN_100GIB_ROOT = 0x2df82ef94d66472dbd46bf76aaa677cf31b2a42447b71f1f82be2a9fb524894b     # seed 0xC0DE, committed whole on one GPU in round 1 (BASELINE.md row 4)
CONFIG1_SLOT_ROOT = 16142339001376051487701717049451130483290782524159378806355159917477338192952      # SURVEY.md 8c
CONFIG1_DATASET_ROOT = 7410604474820069305866101106843319395502234157925946588762357169176803727431


def run_extras(args, torch, dist, pkg, ctx, comm, stream, rank, world, weak_value, timed, barrier) -> dict:
    dataset = importlib.import_module(PKG + ".dataset")
    capi = pkg.capi
    out = {}

    if world == 1:
        # ---- BASELINE configs[0]: eleven 4 MiB fake-data slots, one call, roots read back once ----
        seeds = [dataset.slot_seed(12345, k) for k in range(11)]
        ctx.slots_commit_batch_fake(seeds, 2048)
        t0 = time.perf_counter()
        roots = ctx.slots_commit_batch_fake(seeds, 2048)
        dset_root = ctx.merkle_root(roots)
        t_batch = time.perf_counter() - t0
        assert roots[3] == CONFIG1_SLOT_ROOT and dset_root == CONFIG1_DATASET_ROOT, "config 1 roots differ from the pinned values"
        t0 = time.perf_counter()
        for sd in seeds:
            with ctx.slot_commit_fake(sd, 2048) as s1:
                _ = s1.root
        t_serial = time.perf_counter() - t0
        # ---- 1000 x 4 MiB synthetic slots: batched vs one by one (data resident) ----
        n_small, small_bytes = 1000, 4 << 20
        d_many = torch.empty(n_small * small_bytes, dtype=torch.uint8, device="cuda")
        for k in range(n_small):
            ctx.fill_synthetic_dev(dataset.slot_seed(SEED, k), 0, small_bytes, d_many.data_ptr() + k * small_bytes)
        torch.cuda.synchronize()
        sizes = [small_bytes] * n_small
        ctx.slots_commit_batch_dev(d_many.data_ptr(), sizes)
        t0 = time.perf_counter()
        broots = ctx.slots_commit_batch_dev(d_many.data_ptr(), sizes)
        t_b = time.perf_counter() - t0
        t0 = time.perf_counter()
        sroots = []
        for k in range(100):
            with ctx.slot_commit_dev(d_many.data_ptr() + k * small_bytes, small_bytes) as s1:
                sroots.append(s1.root)
        t_s = (time.perf_counter() - t0) * n_small / 100
        assert broots[:100] == sroots, "batched and one-by-one roots differ"
        out["small_slots"] = {
            "config1_11x4MiB_fake": {"batched_ms": 1e3 * t_batch, "one_by_one_ms": 1e3 * t_serial, "slot_root_3": hex(roots[3]), "dataset_root": hex(dset_root),
                                     "roots_match_pinned_values": True, "api": "cdx_slots_commit_batch_fake + cdx_merkle_root_host",
                                     "note": "includes generating the reference's fake data on the device (sequential per cell)"},
            "batch_1000x4MiB": {"GB_per_s": n_small * small_bytes / t_b / 1e9, "ms": 1e3 * t_b, "one_by_one_GB_per_s": n_small * small_bytes / t_s / 1e9,
                                "one_by_one_ms_extrapolated_from_100": 1e3 * t_s, "api": "cdx_slots_commit_batch_dev", "roots_equal_one_by_one": True,
                                "timing": "wall clock around the call incl. the read-back of 1000 roots; data resident"},
        }
        del d_many
        torch.cuda.empty_cache()
        return out

    # ---- BASELINE configs[3]: ONE 100 GiB slot split over the ranks (strong scaling) ----
    n_total = (100 << 30) // BLOCK
    T, ranges = capi.plan_block_ranges(n_total, world)
    first, count = ranges[rank]
    d = torch.empty(max(count, 1) * BLOCK, dtype=torch.uint8, device="cuda")
    ctx.fill_synthetic_dev(SEED, first * (BLOCK // 8), count * BLOCK, d.data_ptr())
    torch.cuda.synchronize()

    def commit_100g():
        sh = ctx.slot_commit_sharded_dev(comm, d.data_ptr(), count * BLOCK, CELL, BLOCK, first, n_total, T)
        r = sh.root
        sh.free()
        return r
    commit_100g()
    ev_s, wall_s, root100 = timed(commit_100g, 2)
    gbs = n_total * BLOCK * 2 / ev_s / 1e9
    assert root100 == KNOWN_100GIB_ROOT, "100 GiB sharded root differs from the known single-GPU root"
    out["config4_strong"] = {"workload": f"single 100 GiB synthetic slot ({n_total} blocks) split over {world} GPUs, exchange level {T}",
                             "ms_per_step": 1e3 * ev_s / 2, "GB_per_s": gbs, "per_gpu_GB_per_s": gbs / world,
                             "efficiency_vs_weak_per_gpu_rate": (gbs / world) / (weak_value / world), "slot_root": hex(root100),
                             "root_equals_known_single_gpu_root": True, "steps": 2, "warmup": 1, "api": "cdx_slot_commit_sharded_dev + cdx_slot_root",
                             "timing": "CUDA events on the library stream, barrier + synchronize on both sides, max over ranks"}
    del d
    torch.cuda.empty_cache()

    # ---- sharded == whole: rank 0 commits the whole N x 10 GiB slot of the headline alone (tiled generation, no slot-sized buffer) ----
    weak_bytes = int(args.slot_gib * (1 << 30)) // BLOCK * BLOCK * world
    whole_root, t_whole = None, None
    if rank == 0 and args.total_gib <= 0:
        t0 = time.perf_counter()
        with ctx.dataset_commit(None, [(capi.SRC_SYNTHETIC, SEED, weak_bytes)]) as ds1:
            whole_root = ds1.slot_roots[0]
        t_whole = time.perf_counter() - t0
    barrier()
    if rank == 0 and whole_root is not None:
        out["sharded_root_check"] = {"whole_slot_bytes": weak_bytes, "whole_slot_root_one_gpu": hex(whole_root), "one_gpu_s": t_whole,
                                     "api": "cdx_dataset_commit (one synthetic slot, one GPU, tiled generation)"}   # compared with the headline root by the caller

    # ---- BASELINE configs[4]: dataset of 250 slots, mixed sizes, non-power-of-two count ----
    if args.config5 == "on" or (args.config5 == "auto" and world == 8):
        scale = args.config5_scale
        blocks = dataset.draw_slot_blocks(args.config5_slots, scale * (1 << 30), scale * (100 << 30), 12345, pow2_slot=3, pow2_blocks=1 << 15)
        descs = dataset.synthetic_descs(blocks, 12345)
        barrier()
        t0 = time.perf_counter()
        ds = ctx.dataset_commit(comm, descs, keep_slot=3)
        barrier()
        t_commit = time.perf_counter() - t0
        t1 = time.perf_counter()
        idx, paths, leaves = ds.prove(1234567, 100, 32)
        t_prove = time.perf_counter() - t1
        stats = ds.stats
        tt = torch.tensor([t_commit, t_prove, float(stats["bytes_local"])], dtype=torch.float64, device="cuda")
        mx = tt.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        mn = tt.clone()
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        total_b = sum(blocks) * BLOCK
        ok = True
        # two-stage check of every sampled path on the GPU: block level, then slot level (Slot.hs:189-217)
        if rank == 0:
            blk = ctx.reconstruct_roots(leaves, [ci % 32 for ci in idx], 32, paths, depth=5)
            top = ctx.reconstruct_roots(blk, [ci // 32 for ci in idx], blocks[3], [p[5:] for p in paths], depth=15)
            ok = all(t == ds.slot_roots[3] for t in top)
        out["config5"] = {"workload": f"dataset of {len(blocks)} synthetic slots, {scale:g}-{100 * scale:g} GiB log-uniform (seed 12345), slot 3 forced to 2 GiB and sampled",
                          "bytes": total_b, "commit_s": float(mx[0]), "GB_per_s": total_b / float(mx[0]) / 1e9, "prove_100_samples_ms": 1e3 * float(mx[1]),
                          "dataset_root": hex(ds.root), "slot_proof_depth": 8, "all_100_paths_reconstruct_slot_root": bool(ok),
                          "per_rank_bytes_max_over_min": float(mx[2]) / max(float(mn[2]), 1.0), "rank0_stats": stats,
                          "api": "cdx_dataset_commit + cdx_dataset_prove (LPT packing, batching, sharding, root exchange inside the library)",
                          "timing": "wall clock, barrier on both sides, max over ranks; synthetic bytes generated on the device inside the timed region"}
        ds.free()
    return out


if __name__ == "__main__":
    main()
