#!/usr/bin/env python3
"""Compile csrc/capi.cu to a cubin and print, for every S-box loop of a kernel, the FMA-heavy slots H (a 32x32->64
product counts 2) and the other instructions A -- the two terms of the cost model in DESIGN.md section 4.
usage: sass_stats.py [--max-wide N] [kernel-name-substring = k_hash_cells_tma] [extra nvcc flags...]"""
import collections, os, re, subprocess, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
args = sys.argv[1:]
max_wide = 400
if "--max-wide" in args:                      # also report bodies holding several S-boxes (the external-round body has three)
    i = args.index("--max-wide")
    max_wide = int(args[i + 1])
    del args[i:i + 2]
kern = args[0] if args else "k_hash_cells_tma"
extra = args[1:]
src = os.path.join(ROOT, "codex-storage-proofs-circuits_b200", "csrc", "capi.cu")
with tempfile.TemporaryDirectory(prefix="sass_stats_") as out:       # the cubin is scratch: nothing is written into the tree
    cubin = os.path.join(out, "capi.cubin")
    subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-cubin", "-o", cubin, src,
                    "-I", os.path.join(ROOT, "include")] + extra, check=True)
    sass = subprocess.run(["cuobjdump", "-sass", cubin], check=True, capture_output=True, text=True).stdout
cur, funcs = None, collections.OrderedDict()
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1); funcs[cur] = []; continue
    m = re.match(r"^\s+/\*([0-9a-f]{4,6})\*/\s+(.*?);", line)
    if m and cur:
        funcs[cur].append((int(m.group(1), 16), m.group(2)))
for name, ins in funcs.items():
    if kern not in name:
        continue
    print(name, len(ins), "instructions")
    loops = []
    for a, t in ins:
        if "BRA" in t:
            m = re.search(r"0x([0-9a-f]+)", t)
            if m and int(m.group(1), 16) < a:
                loops.append((int(m.group(1), 16), a))
    for s, e in loops:
        c = collections.Counter()
        for a, t in ins:
            if s <= a <= e:
                p = t.split()
                c[p[1] if p[0].startswith("@") else p[0]] += 1
        wide = sum(v for k, v in c.items() if k.startswith("IMAD.WIDE") or k.startswith("IMAD.HI") or k.startswith("UIMAD.WIDE"))
        if wide < 200 or wide > max_wide:
            continue
        other_fma = sum(v for k, v in c.items() if k.startswith("IMAD") and not (k.startswith("IMAD.WIDE") or k.startswith("IMAD.HI")))
        total = sum(c.values())
        H = 2 * wide + other_fma
        A = total - wide - other_fma
        print(f"  loop {s:#x}-{e:#x}: {total} instr, wide products {wide}, other FMA-pipe {other_fma}, H = {H}, A = {A}, H + 0.28 A = {H + 0.28 * A:.0f}")
        print("    ", ", ".join(f"{k} {v}" for k, v in c.most_common(16)))
