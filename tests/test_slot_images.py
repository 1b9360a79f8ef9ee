"""Slot images (cdx_slot_export / cdx_slot_import) against images built by the oracle, without the library.

CPU part: the import-time header checks (csrc/slot_image.h) compiled with g++, plain and under UBSan, against a Python
restatement of them: every single-field mutation of valid headers, shapes, depths at and beyond the path-plan limits,
node counts, lengths, and headers whose 64-bit sizes wrap -- among them headers the previous import accepted.

GPU part: export equals the oracle image byte for byte; an oracle-built image imports and answers like the oracle; the
header table gives the same statuses through cdx_slot_import; every corrupted payload is refused with the exact (tree,
level, node) it breaks; the context keeps working after many refused imports; all of it again within guard bands."""
import ctypes as C
import os
import random
import re
import struct
import subprocess
import sys

import pytest

from conftest import ROOT
from oracle import coracle, pyoracle

gpu = pytest.mark.gpu
R = 21888242871839275222246405745257275088548364400416034343698204186575808495617
M64 = 1 << 64
HEADER = struct.Struct("<8s5Q2I")                 # magic, cell, block, n_blocks, forest_nodes, top_nodes, block_depth, slot_depth
MAX_BLOCK_DEPTH, MAX_SLOT_DEPTH = 32, 39
OK, ARG, SIZE, RANGE, MISMATCH = 0, -1, -2, -4, -8

# (cell, block): cpb 1, 2, 32 and 256; 64-byte and larger multiple-of-32 cells take the TMA sponge, 36 and 100 the plain one
GEOMETRIES = [(64, 64), (36, 36), (64, 128), (100, 200), (64, 2048), (36, 1152), (64, 16384), (100, 25600)]
GEOMETRY_IDS = [f"{c}x{b}" for c, b in GEOMETRIES]


# ---- the oracle's images ----------------------------------------------------------------------------------------

class Chain:
    """the retained levels of an image bottom up, as the import check walks them: a full image's block-forest levels
    0..block_depth, then slot levels 1..slot_depth; a compact image's slot levels 0..slot_depth.  Each level:
    [tree, level, nodes, bottom, singles] -- bottom and singles are the node rule that builds it from the level below."""

    def __init__(self, data, cell, block, kind):
        self.cell, self.block, self.kind = cell, block, kind
        self.cpb = block // cell
        self.n_blocks = len(data) // block
        root, bh, ch = coracle.commit_slot(bytes(data), cell, block, want_cells=True)
        trees = [coracle.merkle_layers(ch[b * self.cpb:(b + 1) * self.cpb]) for b in range(self.n_blocks)]
        slot = coracle.merkle_layers(bh)
        self.root, self.block_depth, self.slot_depth = root, len(trees[0]) - 1, len(slot) - 1
        assert slot[-1] == [root]
        self.levels = []
        if kind == "full":
            for lvl in range(self.block_depth + 1):
                self.levels.append([0, lvl, [v for t in trees for v in t[lvl]], int(lvl == 1), int(self.cpb == 1 and lvl == 1)])
            assert self.levels[-1][2] == bh
        else:
            self.levels.append([1, 0, list(slot[0]), 0, 0])
        for lvl in range(1, self.slot_depth + 1):
            self.levels.append([1, lvl, list(slot[lvl]), int(lvl == 1), 0])

    def header(self, **over):
        f = dict(magic=b"CDXSLOT1" if self.kind == "full" else b"CDXSLOTC", cell=self.cell, block=self.block, n_blocks=self.n_blocks,
                 forest=sum(len(lv[2]) for lv in self.levels if lv[0] == 0),
                 top=sum(len(lv[2]) for lv in self.levels if lv[0] == 1 and lv[1] > 0), bd=self.block_depth, sd=self.slot_depth)
        f.update(over)
        return HEADER.pack(f["magic"], f["cell"], f["block"], f["n_blocks"], f["forest"], f["top"], f["bd"], f["sd"])

    def payload(self):
        return b"".join(v.to_bytes(32, "little") for lv in self.levels for v in lv[2])

    def image(self):
        return self.header() + self.payload()

    def copy(self):
        c = object.__new__(Chain)
        c.__dict__.update(self.__dict__)
        c.levels = [[t, l, list(n), b, s] for t, l, n, b, s in self.levels]
        return c

    # the import check restated: the smallest bad key among the nodes a mutation touched and their parents
    def parent(self, k, i):
        if k + 1 == len(self.levels):
            return None
        return (k + 1, i if self.levels[k + 1][4] else i // 2)

    def node_ok(self, k, i):
        """-> None, 0 (not canonical) or 1 (does not hash from its children)"""
        tree, lvl, nodes, bottom, singles = self.levels[k]
        v = nodes[i]
        if v >= R:
            return 0
        if k == 0:
            return None
        c = self.levels[k - 1][2]                            # the kernels read any 256-bit child mod r
        if singles:
            h = coracle.compress(c[i] % R, 0, 3)
        elif 2 * i + 1 < len(c):
            h = coracle.compress(c[2 * i] % R, c[2 * i + 1] % R, bottom)
        else:
            h = coracle.compress(c[2 * i] % R, 0, bottom + 2)
        return None if h == v else 1

    def first_bad(self, touched):
        cand = set()
        for k, i in touched:
            cand.add((k, i))
            p = self.parent(k, i)
            if p:
                cand.add(p)
        bad = [(k, i, r) for k, i in cand for r in [self.node_ok(k, i)] if r is not None]
        return min(bad, key=lambda b: (b[0], b[1], b[2])) if bad else None

    def message(self, bad):
        k, i, r = bad
        tree, lvl = self.levels[k][:2]
        return f"slot image: {'slot-tree' if tree else 'block-forest'} level {lvl} node {i} " + \
            ("is not canonical" if r == 0 else "does not hash from its children")


def oracle_image(data, cell, block, kind):
    """the image of the slot over `data` as the oracle builds it: header, then the retained levels bottom up"""
    return Chain(data, cell, block, kind).image()


def test_oracle_image_against_pyoracle():
    """the image builder's levels come from the C oracle; at a small geometry they equal the pure-Python oracle's"""
    cell, block, n_blocks = 64, 128, 3
    data = random.Random(5).randbytes(n_blocks * block)
    cells = [pyoracle.hash_cell(data[i * cell:(i + 1) * cell], cell) for i in range(n_blocks * 2)]
    trees = [pyoracle.merkle_layers(cells[2 * b:2 * b + 2]) for b in range(n_blocks)]
    slot = pyoracle.merkle_layers([t[-1][0] for t in trees])
    forest = [v for lvl in range(2) for t in trees for v in t[lvl]]
    top = [v for lv in slot[1:] for v in lv]
    pack = lambda xs: b"".join(v.to_bytes(32, "little") for v in xs)
    full, compact = oracle_image(data, cell, block, "full"), oracle_image(data, cell, block, "compact")
    assert full == HEADER.pack(b"CDXSLOT1", cell, block, n_blocks, len(forest), len(top), 1, 2) + pack(forest + top)
    assert compact == HEADER.pack(b"CDXSLOTC", cell, block, n_blocks, 0, len(top), 1, 2) + pack(slot[0] + top)
    ch = Chain(data, cell, block, "full")
    assert ch.first_bad([(k, i) for k, lv in enumerate(ch.levels) for i in range(len(lv[2]))]) is None


# ---- the header checks, restated ----------------------------------------------------------------------------------

def widths(n):
    w, out = n, [n]
    while len(out) == 1 or w > 1:
        w = (w + 1) // 2
        out.append(w)
    return out


def layout_ref(h, image_bytes):
    """slot_image_layout restated with unbounded integers -> (status, layout or None)"""
    if image_bytes < HEADER.size:
        return SIZE, None
    magic, cell, block, n_blocks, forest_h, top_h, bd_h, sd_h = HEADER.unpack(h)
    if magic not in (b"CDXSLOT1", b"CDXSLOTC"):
        return ARG, None
    compact = magic == b"CDXSLOTC"
    n_bytes = n_blocks * block
    if n_bytes >= M64:
        return SIZE, None
    if cell == 0 or cell % 4 or cell > 1 << 30 or block == 0 or block % cell:
        return SIZE, None
    cpb = block // cell
    if cpb & (cpb - 1) or n_bytes == 0:
        return SIZE, None
    n_cells = n_blocks * cpb
    bd = 1 if cpb == 1 else cpb.bit_length() - 1
    sw = widths(n_blocks)
    sd = len(sw) - 1
    if (bd_h, sd_h) != (bd, sd):
        return ARG, None
    if bd > MAX_BLOCK_DEPTH or sd > MAX_SLOT_DEPTH:
        return RANGE, None
    fw = [n_cells if cpb == 1 else n_cells >> lvl for lvl in range(bd + 1)]
    forest = 0 if compact else sum(fw)
    if forest >= M64:
        return SIZE, None
    if forest_h != forest:
        return ARG, None
    top = sum(sw[1:])
    level0 = sw[0] if compact else forest
    length = HEADER.size + 32 * (level0 + top)
    if top_h != top or length >= M64 or length != image_bytes:
        return SIZE, None
    out = [int(compact), cell, block, n_blocks, n_bytes, n_cells, cpb, bd, sd, forest, top, level0]
    return OK, out + (fw + [0] * 33)[:33] + (sw + [0] * 40)[:40]


def old_import_accepts(h, image_bytes):
    """the import this change replaces, restated with its 64-bit wrapping arithmetic: did it accept the header?"""
    if image_bytes < HEADER.size:
        return False
    magic, cell, block, n_blocks, forest_h, top_h, bd_h, sd_h = HEADER.unpack(h)
    if magic not in (b"CDXSLOT1", b"CDXSLOTC"):
        return False
    compact = magic == b"CDXSLOTC"
    n_bytes = n_blocks * block % M64
    if cell == 0 or cell % 4 or cell > 1 << 30 or block == 0 or block % cell or (block // cell) & (block // cell - 1):
        return False
    if n_bytes == 0 or n_bytes % block or n_blocks == 0:
        return False
    cpb = block // cell
    n_cells = n_blocks * cpb % M64
    bd = 1 if cpb == 1 else (cpb - 1).bit_length()
    sw = widths(n_blocks)
    forest = n_blocks if compact else sum(n_cells if cpb == 1 else n_cells >> lvl for lvl in range(bd + 1)) % M64
    if (0 if compact else forest) != forest_h or (bd, len(sw) - 1) != (bd_h, sd_h):
        return False
    level0 = sw[0] if compact else forest_h
    return sum(sw[1:]) % M64 == top_h and image_bytes == (HEADER.size + 32 * (level0 + top_h)) % M64


def old_consistent(kind, cell, block, n_blocks):
    """the header the old import expected for this geometry, and the (wrapped) image length it wanted"""
    cpb = block // cell
    n_cells = n_blocks * cpb % M64
    bd = 1 if cpb == 1 else (cpb - 1).bit_length()
    sw = widths(n_blocks)
    forest = 0 if kind == "compact" else sum(n_cells if cpb == 1 else n_cells >> lvl for lvl in range(bd + 1)) % M64
    top = sum(sw[1:]) % M64
    level0 = sw[0] if kind == "compact" else forest
    h = HEADER.pack(b"CDXSLOTC" if kind == "compact" else b"CDXSLOT1", cell, block, n_blocks, forest, top, bd, len(sw) - 1)
    return h, (HEADER.size + 32 * (level0 + top)) % M64


def true_header(kind, cell, block, n_blocks, /, **over):
    """the consistent header of a geometry and its image length, from unbounded integers"""
    cpb = block // cell
    bd = 1 if cpb == 1 else cpb.bit_length() - 1
    sw = widths(n_blocks)
    forest = 0 if kind == "compact" else sum(n_blocks * cpb if cpb == 1 else (n_blocks * cpb) >> lvl for lvl in range(bd + 1))
    f = dict(magic=b"CDXSLOTC" if kind == "compact" else b"CDXSLOT1", cell=cell, block=block, n_blocks=n_blocks, forest=forest,
             top=sum(sw[1:]), bd=bd, sd=len(sw) - 1)
    f.update(over)
    length = HEADER.size + 32 * ((n_blocks if kind == "compact" else forest) + sum(sw[1:]))
    return HEADER.pack(f["magic"], f["cell"], f["block"], f["n_blocks"] % M64, f["forest"] % M64, f["top"] % M64, f["bd"] % 2**32, f["sd"] % 2**32), length


def wrap_family():
    """n_blocks = 2^59 + k at cpb 1 and 256, both kinds: every header the old import accepted from a file under 1 MiB"""
    fam = []
    for kind in ("full", "compact"):
        for cell, block in ((4, 4), (4, 1024)):
            for k in range(64):
                h, length = old_consistent(kind, cell, block, (1 << 59) + k)
                if length < 1 << 20 and old_import_accepts(h, length):
                    fam.append((f"wrap-{kind}-cpb{block // cell}-2^59+{k}", h, length, RANGE if block == cell else SIZE))
    return fam


def header_cases():
    """(name, header, image_bytes, pinned status, or None where the restatement decides: a mutated cell or block size can
    describe another valid geometry -- a compact image does not depend on the cell size at one cell per block)"""
    cases = []
    for kind in ("full", "compact"):
        for cell, block in ((64, 64), (64, 128), (64, 2048), (36, 9216)):
            for n_blocks in (1, 13):
                cpb = block // cell
                h, length = true_header(kind, cell, block, n_blocks)
                mag = HEADER.unpack(h)
                name = f"{kind}-cpb{cpb}-{n_blocks}b"
                cases.append((name + "-valid", h, length, OK))
                mut = lambda **o: true_header(kind, cell, block, n_blocks, **o)[0]
                bd, sd, forest, top = mag[6], mag[7], mag[4], mag[5]
                cases += [
                    (name + "-magic", mut(magic=b"CDXSLOTX"), length, ARG),
                    (name + "-magic-case", mut(magic=mag[0].lower()), length, ARG),
                    (name + "-cell0", mut(cell=0), length, SIZE),
                    (name + "-cell6", mut(cell=6, block=6 * cpb), length, SIZE),
                    (name + "-cell-big", mut(cell=(1 << 30) + 4, block=((1 << 30) + 4) * cpb), length, SIZE),
                    (name + "-cell+4", mut(cell=cell + 4), length, SIZE),
                    (name + "-cell/2", mut(cell=cell // 2), length, None),
                    (name + "-cpb3", mut(block=3 * cell), length, SIZE),
                    (name + "-block0", mut(block=0), length, SIZE),
                    (name + "-block*2", mut(block=2 * block), length, None),
                    (name + "-n_blocks0", mut(n_blocks=0), length, SIZE),
                    (name + "-n_blocks+1", mut(n_blocks=n_blocks + 1), length, None),
                    (name + "-n_blocks-1", mut(n_blocks=n_blocks - 1), length, SIZE if n_blocks == 1 else None),
                    (name + "-bd+1", mut(bd=bd + 1), length, ARG),
                    (name + "-bd-1", mut(bd=bd - 1), length, ARG),
                    (name + "-sd+1", mut(sd=sd + 1), length, ARG),
                    (name + "-sd-1", mut(sd=sd - 1), length, ARG),
                    (name + "-forest+1", mut(forest=forest + 1), length, ARG),
                    (name + "-top+1", mut(top=top + 1), length, SIZE),
                    (name + "-top-1", mut(top=top - 1), length, SIZE),
                    (name + "-len+32", h, length + 32, SIZE),
                    (name + "-len-32", h, length - 32, SIZE),
                    (name + "-len55", h, 55, SIZE),
                    (name + "-len0", h, 0, SIZE),
                ]
                if kind == "full":
                    cases.append((name + "-forest-1", mut(forest=forest - 1), length, ARG))
                    cases.append((name + "-forest0", mut(forest=0), length, ARG))
                else:
                    cases.append((name + "-forest-of-full", mut(forest=HEADER.unpack(true_header("full", cell, block, n_blocks)[0])[4]), length, ARG))
        # depths at the path-plan limits, and one past them
        bd_limit = (4, 4 << 32, 1)                       # cpb 2^32: block depth 32
        cases.append((f"{kind}-bd32", *true_header(kind, *bd_limit), OK))
        cases.append((f"{kind}-bd33", *true_header(kind, 4, 4 << 33, 1), RANGE))
        for d in (-1, 1):
            cases.append((f"{kind}-bd32{d:+d}", true_header(kind, *bd_limit, bd=32 + d)[0], true_header(kind, *bd_limit)[1], ARG))
        cases.append((f"{kind}-sd39", *true_header(kind, 4, 4, 1 << 39), OK))
        cases.append((f"{kind}-sd39-ragged", *true_header(kind, 4, 4, (1 << 38) + 1), OK))
        cases.append((f"{kind}-sd40", *true_header(kind, 4, 4, (1 << 39) + 1), RANGE))
        for d in (-1, 1):
            cases.append((f"{kind}-sd39{d:+d}", true_header(kind, 4, 4, 1 << 39, sd=39 + d)[0], true_header(kind, 4, 4, 1 << 39)[1], ARG))
        # sizes that wrap 64 bits inside the depth limits: only the overflow checks refuse these
        for name, geo in (("n_bytes", (4 << 28, 4 << 60, 5)), ("n_bytes-2^39", (4, 4 << 32, (1 << 39) - 1)), ("length", (4, 4 << 32, (1 << 26) + 1))):
            h, length = old_consistent(kind, *geo)
            if kind == "full" or name != "length":
                cases.append((f"{kind}-wrap-{name}", h, length, SIZE))
    cases.append(("issue-compact-1976", HEADER.pack(b"CDXSLOTC", 4, 4, (1 << 59) + 1, 0, (1 << 59) + 59, 1, 60), 1976, RANGE))
    cases.append(("issue-full-2008", HEADER.pack(b"CDXSLOT1", 4, 4, (1 << 59) + 1, (1 << 60) + 2, (1 << 59) + 59, 1, 60), 2008, RANGE))
    return cases + wrap_family()


CASES = header_cases()


def test_header_table_is_what_it_claims():
    """the restatement pins every case; the wraparound headers were accepted by the import this replaces"""
    names = [c[0] for c in CASES]
    assert len(names) == len(set(names))
    for name, h, n, pinned in CASES:
        st, _ = layout_ref(h, n)
        assert n < M64, name
        if pinned is not None:
            assert st == pinned, name
        if "wrap" in name or name.startswith("issue"):
            assert old_import_accepts(h, n), name
    fam = wrap_family()
    for kind in ("full", "compact"):
        for cpb in (1, 256):
            assert any(n.startswith(f"wrap-{kind}-cpb{cpb}-") for n, *_ in fam), (kind, cpb)
    assert {("issue-compact-1976", 1976), ("issue-full-2008", 2008)} <= {(n, l) for n, _, l, _ in CASES}
    assert any(n == "wrap-compact-cpb1-2^59+1" and l == 1976 for n, _, l, _ in fam)
    assert any(n == "wrap-full-cpb1-2^59+1" and l == 2008 for n, _, l, _ in fam)


def _build(tmp_path_factory, name, flags):
    out = str(tmp_path_factory.mktemp(name) / f"lib{name}.so")
    src = os.path.join(ROOT, "tests", "host_emul", "slot_image_check.cpp")
    res = subprocess.run(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-shared", "-fPIC"] + flags + ["-o", out, src],
                         capture_output=True, text=True)
    return res, out


@pytest.fixture(scope="module")
def validator(tmp_path_factory):
    res, out = _build(tmp_path_factory, "imgcheck", ["-O2"])
    assert res.returncode == 0, res.stderr
    return C.CDLL(out)


@pytest.fixture(scope="module")
def validator_ubsan(tmp_path_factory):
    """the same checks built with -fsanitize=undefined -fno-sanitize-recover: any undefined behaviour on the way aborts"""
    res, out = _build(tmp_path_factory, "imgcheck_ubsan", ["-O1", "-g", "-fsanitize=undefined", "-fno-sanitize-recover=undefined"])
    if res.returncode != 0:
        pytest.skip("this g++ cannot build with -fsanitize=undefined: " + res.stderr[-200:])
    try:
        return C.CDLL(out)
    except OSError as e:
        pytest.skip("the UBSan runtime is not loadable: " + str(e))


def run_table(lib):
    fn = lib.image_layout
    fn.restype = C.c_int
    fn.argtypes = [C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_char_p, C.c_size_t]
    out = (C.c_uint64 * 85)()
    msg = C.create_string_buffer(256)
    for name, h, n, _ in CASES:
        want, layout = layout_ref(h, n)
        got = fn(h, n, out, msg, 256)
        assert got == want, (name, got, want, msg.value)
        if want == OK:
            assert list(out) == layout, name
        else:
            assert msg.value, name


def test_header_checks(validator):
    run_table(validator)


def test_header_checks_under_ubsan(validator_ubsan):
    run_table(validator_ubsan)


# ---- GPU: the library against the oracle's images -----------------------------------------------------------------

def random_bytes(seed, n):
    return random.Random(seed).randbytes(n)


def raw_import(ctx, image):
    """cdx_slot_import -> (status, message, handle or None)"""
    h = C.c_void_p()
    rc = ctx.lib.cdx_slot_import(ctx.h, C.cast(C.c_char_p(image), C.c_void_p).value, len(image), C.byref(h))
    return rc, ctx.lib.cdx_last_error(ctx.h).decode(), h


def expect_refused(ctx, image, status, message=None):
    rc, msg, h = raw_import(ctx, image)
    if rc == OK:                                   # never use a handle that should not exist
        ctx.lib.cdx_slot_free(h)
        pytest.fail(f"import accepted an image it should refuse with {status} ({message})")
    assert rc == status, msg
    if message is not None:
        assert msg == message


@gpu
@pytest.mark.parametrize("cell,block", GEOMETRIES, ids=GEOMETRY_IDS)
def test_export_equals_oracle_image(pkg, ctx, tmp_path, cell, block):
    for n_blocks in (1, 2, 3, 5, 8, 13):
        n_bytes = n_blocks * block
        seed = 7919 * n_blocks + cell
        host = random_bytes(seed, n_bytes)
        path = str(tmp_path / f"slot{n_blocks}.dat")
        with open(path, "wb") as f:
            f.write(host)
        fake = ctx.fake_cells(seed, 0, n_bytes // cell, cell)
        for data, commit in ((fake, lambda: ctx.slot_commit_fake(seed, n_bytes // cell, cell, block)),
                             (host, lambda: ctx.slot_commit_host(host, cell, block)),
                             (host, lambda: ctx.slot_commit_file(path, n_bytes, 0, cell, block))):
            with commit() as slot:
                assert slot.export() == oracle_image(data, cell, block, "full"), n_blocks
                slot.compact()
                assert slot.export() == oracle_image(data, cell, block, "compact"), n_blocks


@gpu
@pytest.mark.parametrize("cell,block", GEOMETRIES, ids=GEOMETRY_IDS)
def test_oracle_image_imports_and_answers_like_the_oracle(pkg, ctx, cell, block):
    capi = pkg.capi
    for n_blocks in (8, 13):
        n_bytes = n_blocks * block
        host = random_bytes(cell * block + n_blocks, n_bytes)
        full, compact = Chain(host, cell, block, "full"), Chain(host, cell, block, "compact")
        bd, sd, cpb = full.block_depth, full.slot_depth, full.cpb
        n_cells = n_blocks * cpb
        md = bd + sd + 1
        trees = [coracle.merkle_layers(full.levels[0][2][b * cpb:(b + 1) * cpb]) for b in range(n_blocks)] if cpb > 1 else \
            [coracle.merkle_layers([v]) for v in full.levels[0][2]]
        slot_layers = [lv[2] for lv in compact.levels]

        def want_path(i):
            merged = pyoracle.merge_merkle_proofs(pyoracle.merkle_proof(trees[i // cpb], i % cpb), pyoracle.merkle_proof(slot_layers, i // cpb))
            return pyoracle.pad_merkle_proof(merged, md).merkle_path, merged.leaf_value

        with ctx.slot_import(full.image()) as s:
            assert s.root == full.root and s.shape == (n_cells, n_blocks, bd, sd)
            for k in range(bd + 1):
                assert s.read_layer(0, k, 0, len(full.levels[k][2])) == full.levels[k][2]
            for k in range(sd + 1):
                assert s.read_layer(1, k, 0, len(slot_layers[k])) == slot_layers[k]
            paths, leaves = s.cell_paths(list(range(n_cells)), md)
            for i in range(n_cells):
                assert (paths[i], leaves[i]) == want_path(i), i
            if n_blocks == 8:
                entropies = [3, R - 1]
                idx, ps, ls = s.prove_batch(entropies, 10, md)
                for e, row_i, row_p, row_l in zip(entropies, idx, ps, ls):
                    assert row_i == [coracle.cell_index(e, full.root, n_cells, c) for c in range(1, 11)]
                    assert [(p, l) for p, l in zip(row_p, row_l)] == [want_path(i) for i in row_i]
        with ctx.slot_import(compact.image()) as s:
            assert s.root == compact.root and s.shape == (n_cells, n_blocks, bd, sd)
            assert s.read_layer(0, bd, 0, n_blocks) == slot_layers[0]
            for k in range(sd + 1):
                assert s.read_layer(1, k, 0, len(slot_layers[k])) == slot_layers[k]
            if n_blocks == 8:
                entropies = [3, R - 1]
                idx, ps, ls, cells = s.prove_from_source((capi.SRC_HOST, host, n_bytes), entropies, 10, md)
                for e, row_i, row_p, row_l, row_c in zip(entropies, idx, ps, ls, cells):
                    assert row_i == [coracle.cell_index(e, compact.root, n_cells, c) for c in range(1, 11)]
                    assert [(p, l) for p, l in zip(row_p, row_l)] == [want_path(i) for i in row_i]
                    assert row_c == [host[i * cell:(i + 1) * cell] for i in row_i]


@gpu
def test_header_table_through_import(pkg, ctx):
    """every case of the CPU table whose image is small enough to build: the same status from cdx_slot_import.  Refused
    headers carry zero payloads; the valid small ones carry the oracle's payload"""
    payloads = {}
    run = set()
    for name, h, n, pinned in CASES:
        want, _ = layout_ref(h, n)
        magic, cell, block, n_blocks = HEADER.unpack(h)[:4]
        if n > 1 << 22 or (want == OK and n_blocks * block > 1 << 22):
            continue
        if want == OK:
            key = (magic, cell, block, n_blocks)
            if key not in payloads:
                ch = Chain(random_bytes(n_blocks, n_blocks * block), cell, block, "compact" if magic == b"CDXSLOTC" else "full")
                assert ch.header() == h
                payloads[key] = ch
            with ctx.slot_import(h + payloads[key].payload()) as s:
                assert s.root == payloads[key].root, name
        else:
            image = (h + bytes(max(0, n - HEADER.size)))[:n]
            expect_refused(ctx, image, want)
        run.add(name)
    assert {"issue-compact-1976", "issue-full-2008"} <= run
    assert all(n in run for n, *_ in wrap_family())


def corruption_sites(ch):
    """(level index, node) pairs: first, middle and last node of every level (the last of a ragged level is its odd tail)"""
    return [(k, i) for k, lv in enumerate(ch.levels) for i in sorted({0, len(lv[2]) // 2, len(lv[2]) - 1})]


@gpu
@pytest.mark.parametrize("cell,block", [(64, 64), (64, 128), (36, 1152), (64, 16384)], ids=["cpb1", "cpb2", "cpb32", "cpb256"])
@pytest.mark.parametrize("kind", ["full", "compact"])
def test_corrupted_payloads_are_refused(ctx, cell, block, kind):
    n_blocks = 13                                    # slot levels 13, 7, 4, 2, 1: ragged
    base = Chain(random_bytes(cell + block, n_blocks * block), cell, block, kind)
    with ctx.slot_import(base.image()) as s:
        assert s.root == base.root

    def refused(ch, touched):
        bad = ch.first_bad(touched)
        assert bad is not None
        expect_refused(ctx, ch.image(), MISMATCH, ch.message(bad))
        return bad

    # one flipped bit at every level of both trees
    for k, i in corruption_sites(base):
        ch = base.copy()
        ch.levels[k][2][i] ^= 1 << (i % 250)
        bad = refused(ch, [(k, i)])
        assert bad[:2] == ((k, i) if k > 0 or bad[2] == 0 else ch.parent(k, i))
    # two corrupted nodes: the smaller key is named
    rnd = random.Random(block)
    for _ in range(6):
        (k1, i1), (k2, i2) = rnd.sample(corruption_sites(base), 2)
        ch = base.copy()
        ch.levels[k1][2][i1] ^= 2
        ch.levels[k2][2][i2] ^= 4
        refused(ch, [(k1, i1), (k2, i2)])
    # non-canonical elements: r and 2^256 - 1 at the bottom (their parents would see the same value mod r) and at the root
    for k, i in ((0, 0), (0, len(base.levels[0][2]) - 1), (len(base.levels) - 1, 0)):
        for v in (R, (1 << 256) - 1, base.levels[k][2][i] + R):
            ch = base.copy()
            ch.levels[k][2][i] = v
            assert refused(ch, [(k, i)]) == (k, i, 0)
    # two block hashes swapped: caught where they are hashed
    kb = len(base.levels) - 1 - base.slot_depth          # the block hashes' level in the chain
    ch = base.copy()
    nodes = ch.levels[kb][2]
    nodes[2], nodes[9] = nodes[9], nodes[2]
    bad = refused(ch, [(kb, 2), (kb, 9)])
    assert bad == ((kb + 1, 1, 1) if kind == "compact" else (kb, 2, 1))
    # two sibling subtrees swapped with everything below them: only their common parent is inconsistent
    singles = base.cpb == 1
    for top_k in range(kb, len(base.levels) - 1):
        ch = base.copy()
        for k in range(top_k, -1, -1):                 # the nodes under node 0 and node 1 of chain level top_k: w each
            w = 1 << (top_k - k) if k >= kb else (1 << (top_k - kb)) << (0 if singles else kb - k)
            nodes = ch.levels[k][2]
            if 2 * w > len(nodes):
                break                                  # node 1 is the ragged tail at this height
            nodes[0:w], nodes[w:2 * w] = nodes[w:2 * w], nodes[0:w]
        else:
            assert ch.first_bad([(k, i) for k, lv in enumerate(ch.levels) for i in range(len(lv[2]))]) == (top_k + 1, 0, 1)
            expect_refused(ctx, ch.image(), MISMATCH, ch.message((top_k + 1, 0, 1)))


@gpu
def test_context_survives_refused_imports(ctx):
    cell, block, n_blocks = 64, 2048, 5
    host = random_bytes(77, n_blocks * block)
    base = Chain(host, cell, block, "full")
    image = base.image()
    for k in range(100):
        if k % 2:
            expect_refused(ctx, image[:-32 * (k % 7 + 1)], SIZE)
        else:
            ch = base.copy()
            lv = ch.levels[k % len(ch.levels)][2]
            lv[k % len(lv)] ^= 1 << 7
            rc, msg, h = raw_import(ctx, ch.image())
            if rc == OK:
                ctx.lib.cdx_slot_free(h)
                pytest.fail("a corrupted image was accepted")
            assert rc == MISMATCH, msg
    with ctx.slot_commit_host(host, cell, block) as s:
        assert s.root == base.root and s.export() == image
    with ctx.slot_import(image) as s:
        assert s.root == base.root and s.export() == image


@gpu
def test_slot_images_within_guard_bands():
    """every GPU test above again with CODEX_COMMIT_GUARD=1 (4 KiB bands around every device allocation of the library,
    checked when it is freed): no write outside an allocation, refused imports included"""
    env = dict(os.environ, CODEX_COMMIT_GUARD="1")
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-x", "-q", "-k", "not within_guard_bands",
                          "-p", "no:cacheprovider"], capture_output=True, text=True, env=env, timeout=1500, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "CODEX_COMMIT_GUARD" not in res.stderr
    assert re.search(r"\b\d+ passed", res.stdout), res.stdout[-2000:]
