"""The field arithmetic of fr.cuh and the Poseidon2 steps of poseidon2.cuh, bit for bit on RAW limb values, at the edges
of their lazy ranges.

Every op of tests/fr_ops/fr_ops.cuh has an exact closed form over the integers (W = 2^256, B = r + 2^250):
    REDC(t) = (t + ((-t r^-1) mod W) r) / W
    mont_mul(a, b) = REDC(a b)               a < W - r, b < W
    mont_sqr(a)    = REDC(a^2)               a < (W - r) / 2
    reduce_tab(v, carry) = V - floor(floor(V / 2^250) 2^250 / r) r,   V = v + carry W, carry in {0, 1}
and the rest are compositions of these (the references below), so the lazy values are pinned exactly, not modulo r.
Each reference asserts its op's input contract: an input generator that leaves a contract fails here instead of
testing undefined territory (or, for reduce_tab, reading past the 128-row table).

The CPU tests pin the references and the g++ build of the dispatcher (against the C emulation of the PTX primitives,
tests/host_emul/fr_rows_host.h) to each other; the GPU tests pin the sm_100a build to both."""
import ctypes as C
import functools
import importlib
import os
import random
import subprocess

import numpy as np
import pytest

from conftest import PKG, ROOT
from oracle.poseidon2_rc import RC_EXT, RC_INT

HERE = os.path.join(ROOT, "tests", "fr_ops")

R = 21888242871839275222246405745257275088548364400416034343698204186575808495617
W = 1 << 256
B = R + (1 << 250)                     # reduce_tab's output bound
NINV = -pow(R, -1, W) % W
WINV = pow(W, -1, R)
R2 = W * W % R                         # CDX_R2_INIT
ONE = W % R                            # CDX_ONE_INIT
MUL_MAX = W - R                        # mont_mul: a < MUL_MAX
SQR_MAX = (W - R) // 2                 # mont_sqr and sbox: a < SQR_MAX
SBOX_OUT = 164 * R // 100              # documented S-box output bound, the mixes' input range
RC_EXT_M = [[c * W % R for c in rnd] for rnd in RC_EXT]
RC_INT_M = [c * W % R for c in RC_INT]


# ---- exact references --------------------------------------------------------------------------------------

def redc(t):
    return (t + (t * NINV % W) * R) >> 256


def mont_mul(a, b):
    assert 0 <= a < MUL_MAX and 0 <= b < W, (hex(a), hex(b))
    return redc(a * b)


def mont_sqr(a):
    assert 0 <= a < SQR_MAX, hex(a)
    return redc(a * a)


def reduce_tab(v, carry):
    assert 0 <= v < W and carry in (0, 1), (hex(v), carry)
    v += carry * W
    return v - ((v >> 250) << 250) // R * R


def add_reduce(a, b):
    assert 0 <= a < W and 0 <= b < W
    return reduce_tab((a + b) % W, (a + b) >> 256)


def add_lazy(a, b):
    assert a + b < W, (hex(a), hex(b))
    return a + b


def reduce_once(a):
    assert 0 <= a < 2 * R, hex(a)
    return a % R


def add_mod(a, b):
    assert 0 <= a < R and 0 <= b < R
    return (a + b) % R


def dbl_mod(a):
    assert 0 <= a < R
    return 2 * a % R


def to_mont(a):
    assert 0 <= a < W
    return a * W % R


def from_mont(a):
    assert 0 <= a < 2 * R
    return a * WINV % R


def mont_from_u32(c):
    assert 0 <= c < 1 << 32
    return to_mont(c)


def sbox(x):
    return mont_mul(mont_sqr(mont_sqr(x)), x)


def mix_external(x, y, z):
    assert max(x, y, z) < SBOX_OUT                      # S-box outputs, or state words < B
    s = add_lazy(add_lazy(x, y), z)
    return add_reduce(x, s), add_reduce(y, s), add_reduce(z, s)


def mix_internal(x, y, z):
    assert x < SBOX_OUT and max(y, z) < B               # x through its S-box, y and z state words
    s = add_lazy(x, add_lazy(y, z))
    return add_reduce(x, s), reduce_tab(add_lazy(y, s), 0), add_reduce(z, add_lazy(z, s))


def absorb(w, m):
    assert 0 <= w < B
    return add_reduce(w, mont_mul(R2, m))


def absorb_one(w):
    assert 0 <= w < B
    return add_reduce(w, ONE)


def sponge_iv(rate):
    assert 0 <= rate < (1 << 32) - 0x300       # limb 0 is 0x300 + rate
    return to_mont((1 << 64) + 0x300 + rate)


def permute(x, y, z):
    assert max(x, y, z) < B
    x, y, z = mix_external(x, y, z)
    for half in range(2):
        for c in RC_EXT_M[4 * half:4 * half + 4]:
            x, y, z = sbox(add_lazy(x, c[0])), sbox(add_lazy(y, c[1])), sbox(add_lazy(z, c[2]))
            x, y, z = mix_external(x, y, z)
        if half == 0:
            for c in RC_INT_M:
                x = sbox(add_lazy(x, c))
                x, y, z = mix_internal(x, y, z)
    return x, y, z


def compress_keyed(x, y, key):
    return permute(x, y, mont_from_u32(key))[0]


# (name, reference on one record (x, y, z, aux) -> tuple of output words); the order is the FrOp enum of fr_ops.cuh
OPS = [
    ("mont_mul", lambda x, y, z, k: (mont_mul(x, y),)),
    ("mont_sqr", lambda x, y, z, k: (mont_sqr(x),)),
    ("reduce_tab", lambda x, y, z, k: (reduce_tab(x, k),)),
    ("add_reduce", lambda x, y, z, k: (add_reduce(x, y),)),
    ("reduce_once", lambda x, y, z, k: (reduce_once(x),)),
    ("add_mod", lambda x, y, z, k: (add_mod(x, y),)),
    ("dbl_mod", lambda x, y, z, k: (dbl_mod(x),)),
    ("to_mont", lambda x, y, z, k: (to_mont(x),)),
    ("from_mont", lambda x, y, z, k: (from_mont(x),)),
    ("mont_from_u32", lambda x, y, z, k: (mont_from_u32(k),)),
    ("sbox", lambda x, y, z, k: (sbox(x),)),
    ("mix_external", lambda x, y, z, k: mix_external(x, y, z)),
    ("mix_internal", lambda x, y, z, k: mix_internal(x, y, z)),
    ("absorb", lambda x, y, z, k: (absorb(x, y),)),
    ("absorb_one", lambda x, y, z, k: (absorb_one(x),)),
    ("sponge_iv", lambda x, y, z, k: (sponge_iv(k),)),
    ("permute", lambda x, y, z, k: permute(x, y, z)),
    ("compress_keyed", lambda x, y, z, k: (compress_keyed(x, y, k),)),
]
OP_NAMES = [name for name, _ in OPS]
OP_INDEX = {name: i for i, name in enumerate(OP_NAMES)}
SLOW_OPS = ("permute", "compress_keyed")       # 80 S-boxes per record: fewer random records


def reference(name, rec):
    assert all(0 <= w < W for w in rec[:3]) and 0 <= rec[3] < 1 << 32, rec
    out = dict(OPS)[name](*rec)
    return tuple(out) + (0,) * (3 - len(out))


# ---- edge sets (Python ints, exact) --------------------------------------------------------------------------

LIMB_EDGES = [0, 1, (1 << 31) - 1, 1 << 31, (1 << 32) - 2, (1 << 32) - 1]
M32 = (1 << 32) - 1
R0 = R & M32                           # a first-row product with this low limb makes the Montgomery factor 2^32 - 1


def from_limbs(limbs):
    return sum(v << (32 * i) for i, v in enumerate(limbs))


@functools.lru_cache(None)
def limb_patterns():
    """values whose limbs drive carries through 0xffffffff words and sign bits: one limb value everywhere, one limb set
    over an all-zero or all-ones background, alternating all-ones and zero limbs"""
    vals = {from_limbs([v] * 8) for v in LIMB_EDGES}
    for p in range(8):
        for v in LIMB_EDGES:
            for bg in (0, M32):
                limbs = [bg] * 8
                limbs[p] = v
                vals.add(from_limbs(limbs))
    vals.add(from_limbs([M32, 0] * 4))
    vals.add(from_limbs([0, M32] * 4))
    return sorted(vals)


def sqrt_mod_2_32(t):
    """x with x^2 = t mod 2^32 (t = 1 mod 8), by lifting one bit at a time"""
    x = 1
    for i in range(3, 32):                 # x^2 = t mod 2^i  ->  mod 2^(i+1)
        if (x * x - t) >> i & 1:
            x += 1 << (i - 1)
    assert x * x & M32 == t
    return x


def edge_values(bound):
    """every value below `bound` from: the limb patterns, the bound's last values, and k r - 1, k r, k r + 1 for every k
    the bound allows"""
    vals = set(limb_patterns()) | {bound - 1, bound - 2, bound - (1 << 32), bound - (1 << 224)}
    vals |= {k * R + d for k in range(1, bound // R + 2) for d in (-1, 0, 1)}
    return sorted(v for v in vals if 0 <= v < bound)


def with_low_limb(v, l0):
    return v - (v & M32) + l0


def within_contract(name, rec):
    try:
        reference(name, rec)
        return True
    except AssertionError:
        return False


@functools.lru_cache(None)
def edge_records(name):
    """records (x, y, z, aux) at the edges of op `name`'s contract; candidates built from several bounds are clamped to
    the contract by dropping what its reference rejects, and the ones the contract names are asserted present"""
    rnd = random.Random(OP_INDEX[name])
    must = []
    if name == "mont_mul":
        xs, ys = edge_values(MUL_MAX), edge_values(W)
        recs = [(x, y, 0, 0) for x in xs for y in ys]
        # first-row Montgomery factor 2^32 - 1 (a0 b0 = r0 mod 2^32) and 0 (a0 b0 = 0)
        recs += [(x, with_low_limb(y, R0 * pow(x & M32, -1, 1 << 32) & M32), 0, 0) for x in xs if x & 1 for y in ys[::7]]
        recs += [(with_low_limb(x, 1 << 16), with_low_limb(y, 1 << 16), 0, 0) for x in xs[::5] for y in ys[::5]]
        must = [(MUL_MAX - 1, W - 1, 0, 0)]
    elif name in ("mont_sqr", "sbox"):
        xs = edge_values(SQR_MAX) + [B - 1, B + R - 1]               # B + R - 1: the permutation's largest S-box input
        s = sqrt_mod_2_32(R0)                  # the four square roots of r0: first-row factor 2^32 - 1
        roots = [s, -s & M32, s ^ 1 << 31, (-s & M32) ^ 1 << 31]
        xs += [with_low_limb(x, l0) for x in xs[::3] for l0 in roots + [0, 1 << 16]]
        recs = [(x, 0, 0, 0) for x in xs]
        must = [(SQR_MAX - 1, 0, 0, 0)]
    elif name == "reduce_tab":
        # k-major per offset: 32 consecutive records (one warp) fall in 32 different table rows
        vs = [(k << 250) + d for d in (0, -1, 1) for k in range(129)] + [2 * W - 1]
        vs += [v + c * W for v in limb_patterns() for c in (0, 1)]
        recs = [(v % W, 0, 0, v >> 256) for v in vs if 0 <= v < 2 * W]
        must = [(W - 1, 0, 0, 1), (0, 0, 0, 1)]
    elif name == "add_reduce":
        vs = [(k << 250) + d for k in range(129) for d in (-1, 0, 1)] + [2 * W - 2]
        recs = [(a, v - a, 0, 0) for v in vs for a in (min(v, W - 1), v // 2, min(v, R - 1), min(v, B - 1))]
        xs = edge_values(W)[::3]
        recs += [(x, y, 0, 0) for x in xs for y in xs]
        must = [(W - 1, W - 1, 0, 0)]
    elif name == "reduce_once":
        recs = [(x, 0, 0, 0) for x in edge_values(2 * R)]
        must = [(v, 0, 0, 0) for v in (R - 1, R, R + 1, 2 * R - 1)]
    elif name == "add_mod":
        xs = edge_values(R)
        recs = [(x, y, 0, 0) for x in xs for y in xs]
        recs += [(x, R - x + d, 0, 0) for x in xs for d in (-1, 0, 1)]
        must = [(R - 1, R - 1, 0, 0), (1, R - 1, 0, 0)]
    elif name == "dbl_mod":
        recs = [(x, 0, 0, 0) for x in edge_values(R) + [R // 2, R // 2 + 1]]
        must = [(R - 1, 0, 0, 0)]
    elif name == "to_mont":
        recs = [(x, 0, 0, 0) for x in edge_values(W)]
        must = [(v, 0, 0, 0) for v in (0, 1, R - 1, R, W - 1)]
    elif name == "from_mont":
        recs = [(x, 0, 0, 0) for x in edge_values(2 * R)]
        must = [(v, 0, 0, 0) for v in (0, 1, R - 1, R, 2 * R - 1)]
    elif name == "mont_from_u32":
        recs = [(0, 0, 0, k) for k in list(range(4)) + LIMB_EDGES + [R0]]
        must = [(0, 0, 0, k) for k in range(4)]
    elif name in ("mix_external", "mix_internal"):
        small = [0, 1, M32, R - 1, R, R + 1, B - 1, SBOX_OUT - 1] + [rnd.randrange(SBOX_OUT) for _ in range(4)]
        recs = [(x, y, z, 0) for x in small for y in small for z in small]
        must = [(SBOX_OUT - 1, B - 1, B - 1, 0)] if name == "mix_internal" else [(SBOX_OUT - 1,) * 3 + (0,)]
    elif name == "absorb":
        recs = [(w, m, 0, 0) for w in edge_values(B) for m in edge_values(W)[::2]]
        must = [(B - 1, W - 1, 0, 0)]
    elif name == "absorb_one":
        recs = [(w, 0, 0, 0) for w in edge_values(B)]
        must = [(B - 1, 0, 0, 0)]
    elif name == "sponge_iv":
        recs = [(0, 0, 0, k) for k in list(range(4)) + [255, 256, 1 << 31, (1 << 32) - 0x301]]
        must = [(0, 0, 0, 1), (0, 0, 0, 2)]
    elif name == "permute":
        words = [0, 1, R - 1, R, B - 1]
        recs = [(x, y, z, 0) for x in words for y in words for z in words]
        recs += [tuple(rnd.randrange(B) for _ in range(3)) + (0,) for _ in range(16)]
        must = [(B - 1, B - 1, B - 1, 0), (0, 0, 0, 0)]
    elif name == "compress_keyed":
        recs = [(x, y, 0, k) for k in range(4) for x, y in [(0, 0), (B - 1, B - 1), (R - 1, 0), (0, R)]]
        recs += [(rnd.randrange(B), rnd.randrange(B), 0, rnd.randrange(4)) for _ in range(8)]
        must = [(B - 1, B - 1, 0, 3)]
    else:
        raise KeyError(name)
    recs = list(dict.fromkeys(rec for rec in recs if within_contract(name, rec)))
    for rec in must:
        assert rec in recs, (name, rec)
    return recs


# ---- biased random records (numpy limbs) ---------------------------------------------------------------------

LIMB_EDGES_NP = np.array(LIMB_EDGES, dtype=np.uint32)


def to_limbs(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), dtype="<u4").reshape(-1, 8).copy()


def limbs_to_ints(a):
    raw = np.ascontiguousarray(a, dtype="<u4").tobytes()
    return [int.from_bytes(raw[i:i + 32], "little") for i in range(0, len(raw), 32)]


def biased_limbs(rng, n):
    """n x 8 limbs; per row, each limb is an edge value (0, 1, 2^31 - 1, 2^31, 2^32 - 2, 2^32 - 1) with probability
    0, 0.3 or 0.7 and uniform otherwise"""
    uni = rng.integers(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    edge = LIMB_EDGES_NP[rng.integers(0, len(LIMB_EDGES), size=(n, 8))]
    p = rng.choice([0.0, 0.3, 0.7], size=(n, 1))
    return np.where(rng.random((n, 8)) < p, edge, uni)


def _add(a, b):
    out, c = np.empty_like(a), np.zeros(len(a), np.uint64)
    for k in range(8):
        s = a[:, k].astype(np.uint64) + b[:, k] + c
        out[:, k], c = (s & M32).astype(np.uint32), s >> 32
    return out, c


def _sub(a, b):
    out, bw = np.empty_like(a), np.zeros(len(a), np.int64)
    for k in range(8):
        d = a[:, k].astype(np.int64) - b[:, k] - bw
        out[:, k], bw = (d & M32).astype(np.uint32), (d < 0).astype(np.int64)
    return out, bw


def _less(a, bound):
    if bound >= W:
        return np.ones(len(a), bool)
    b = to_limbs([bound])[0]
    lt, decided = np.zeros(len(a), bool), np.zeros(len(a), bool)
    for k in range(7, -1, -1):
        lt |= ~decided & (a[:, k] < b[k])
        decided |= a[:, k] != b[k]
    return lt


def below(rng, n, bound, anchors=()):
    """n x 8 limbs of values < bound: half biased random limbs, half an anchor (bound - 1, or one of `anchors`) plus or
    minus a biased value of 0..7 low limbs; rows that land at or above the bound are drawn again"""
    anc = to_limbs([bound - 1] + [a for a in anchors if a < bound])
    out, todo = np.empty((n, 8), np.uint32), np.arange(n)
    while len(todo):
        m = len(todo)
        d = biased_limbs(rng, m)
        d[np.arange(8)[None, :] >= rng.integers(0, 8, size=(m, 1))] = 0
        a = anc[rng.integers(0, len(anc), size=m)]
        (plus, carry), (minus, borrow) = _add(a, d), _sub(a, d)
        up, near = rng.random(m) < 0.5, rng.random(m) < 0.5
        cand = np.where(near[:, None], np.where(up[:, None], plus, minus), biased_limbs(rng, m))
        ok = ~(near & np.where(up, carry != 0, borrow != 0)) & _less(cand, bound)
        out[todo[ok]] = cand[ok]
        todo = todo[~ok]
    return out


R_MULTIPLES = [k * R for k in range(1, 6)]
TABLE_BOUNDS = [k << 250 for k in range(1, 64)]


def random_records(name, n, seed):
    """(in_ n x 3 x 8 uint32, aux n uint32) inside op `name`'s documented ranges"""
    rng = np.random.default_rng([seed, OP_INDEX[name]])
    words = [np.zeros((n, 8), np.uint32) for _ in range(3)]
    aux = np.zeros(n, np.uint32)
    if name == "mont_mul":
        words[0], words[1] = below(rng, n, MUL_MAX, R_MULTIPLES), below(rng, n, W, R_MULTIPLES)
    elif name in ("mont_sqr", "sbox"):
        words[0] = below(rng, n, SQR_MAX, R_MULTIPLES + [B])
    elif name == "reduce_tab":
        words[0], aux[:] = below(rng, n, W, TABLE_BOUNDS), rng.integers(0, 2, n)
    elif name == "add_reduce":
        words[0], words[1] = below(rng, n, W, TABLE_BOUNDS), below(rng, n, W, TABLE_BOUNDS)
    elif name in ("reduce_once", "from_mont"):
        words[0] = below(rng, n, 2 * R, [R])
    elif name == "add_mod":
        words[0], words[1] = below(rng, n, R), below(rng, n, R)
    elif name == "dbl_mod":
        words[0] = below(rng, n, R, [R // 2 + 1])
    elif name == "to_mont":
        words[0] = below(rng, n, W, R_MULTIPLES)
    elif name == "mont_from_u32":
        aux[:] = biased_limbs(rng, n)[:, 0]
    elif name == "mix_external":
        words = [below(rng, n, SBOX_OUT, [R]) for _ in range(3)]
    elif name == "mix_internal":
        words = [below(rng, n, SBOX_OUT, [R]), below(rng, n, B, [R]), below(rng, n, B, [R])]
    elif name == "absorb":
        words[0], words[1] = below(rng, n, B, [R]), below(rng, n, W, R_MULTIPLES)
    elif name == "absorb_one":
        words[0] = below(rng, n, B, [R])
    elif name == "sponge_iv":
        aux[:] = rng.integers(0, (1 << 32) - 0x300, n)
    elif name == "permute":
        words = [below(rng, n, B, [R]) for _ in range(3)]
    elif name == "compress_keyed":
        words[0], words[1], aux[:] = below(rng, n, B, [R]), below(rng, n, B, [R]), biased_limbs(rng, n)[:, 0]
    else:
        raise KeyError(name)
    return np.ascontiguousarray(np.stack(words, axis=1)), aux


def pack(recs):
    return to_limbs([w for rec in recs for w in rec[:3]]).reshape(-1, 3, 8), np.array([rec[3] for rec in recs], np.uint32)


def unpack(in_, aux):
    w = limbs_to_ints(in_.reshape(-1, 8))
    return [(w[3 * i], w[3 * i + 1], w[3 * i + 2], int(aux[i])) for i in range(len(aux))]


def check_aux(name, aux):
    # a carry above 1 would index past the 128 rows of the reduction table
    assert name != "reduce_tab" or int(aux.max(initial=0)) <= 1


def assert_matches(name, recs, got, want):
    """got, want: n x 3 x 8 limbs; on a mismatch, report the first failing record in hex"""
    bad = np.nonzero((got != want).any(axis=(1, 2)))[0]
    if len(bad):
        i = bad[0]
        fmt = lambda a: [hex(v) for v in limbs_to_ints(a)]
        pytest.fail(f"{name}: {len(bad)} of {len(got)} records differ; first: in {[hex(v) for v in recs[i][:3]]} "
                    f"aux {recs[i][3]}: got {fmt(got[i])}, want {fmt(want[i])}")


def expected(name, recs):
    return to_limbs([w for rec in recs for w in reference(name, rec)]).reshape(-1, 3, 8)


# ---- the two builds of fr_ops.cuh ----------------------------------------------------------------------------

@pytest.fixture(scope="module")
def host_ops(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("fr_ops_host") / "libfrops_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "tests", "host_emul"), "-o", out,
                    os.path.join(HERE, "fr_ops_host.cpp")], check=True)
    lib = C.CDLL(out)
    lib.fr_ops_host.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]

    def run(name, in_, aux):
        check_aux(name, aux)
        in_, aux = np.ascontiguousarray(in_, np.uint32), np.ascontiguousarray(aux, np.uint32)
        out = np.full_like(in_, M32)
        lib.fr_ops_host(OP_INDEX[name], in_.ctypes.data, aux.ctypes.data, out.ctypes.data, len(aux))
        return out
    return run


def build_device_ops(out_dir):
    build = importlib.import_module(PKG + ".build")
    out = os.path.join(out_dir, "libfrops_dev.so")
    res = subprocess.run([build._nvcc()] + build.NVCC_FLAGS + ["-o", out, os.path.join(HERE, "fr_ops.cu")],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    return out


@pytest.fixture(scope="module")
def device_ops(tmp_path_factory):
    import torch
    lib = C.CDLL(build_device_ops(str(tmp_path_factory.mktemp("fr_ops_dev"))))
    lib.fr_ops_launch.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_int)]
    lib.fr_ops_launch.restype = C.c_int

    def run(name, in_, aux, block=256):
        check_aux(name, aux)
        d_in = torch.from_numpy(np.ascontiguousarray(in_, np.uint32).view(np.int32)).cuda()
        d_aux = torch.from_numpy(np.ascontiguousarray(aux, np.uint32).view(np.int32)).cuda()
        d_out = torch.full_like(d_in, -1)
        torch.cuda.synchronize()
        sync_err = C.c_int(-1)
        launch_err = lib.fr_ops_launch(OP_INDEX[name], d_in.data_ptr(), d_aux.data_ptr(), d_out.data_ptr(), len(aux), block,
                                       C.byref(sync_err))
        assert (launch_err, sync_err.value) == (0, 0), (name, block, launch_err, sync_err.value)
        return d_out.cpu().numpy().view(np.uint32)
    return run


N_RANDOM_CPU = 1 << 16
N_RANDOM_GPU = 1 << 20
N_PERM_CPU = 256
N_PERM_GPU = 4096


# ---- CPU: references vs the host build -----------------------------------------------------------------------

@pytest.mark.parametrize("name", OP_NAMES)
def test_host_build_matches_reference_on_edges(host_ops, name):
    recs = edge_records(name)
    in_, aux = pack(recs)
    assert_matches(name, recs, host_ops(name, in_, aux), expected(name, recs))


@pytest.mark.parametrize("name", OP_NAMES)
def test_host_build_matches_reference_on_random(host_ops, name):
    in_, aux = random_records(name, N_PERM_CPU if name in SLOW_OPS else N_RANDOM_CPU, seed=1)
    recs = unpack(in_, aux)
    assert_matches(name, recs, host_ops(name, in_, aux), expected(name, recs))


def test_edge_records_cover_every_table_row():
    """the reduce_tab edge set reaches all 128 rows, and each of its first four warps hits 32 different rows"""
    recs = edge_records("reduce_tab")
    rows = [((k << 256) + v) >> 250 for v, _, _, k in recs]
    assert set(rows) == set(range(128))
    assert all(len(set(rows[w:w + 32])) == 32 for w in range(0, 128, 32))


def test_device_harness_cross_compiles(tmp_path):
    build = importlib.import_module(PKG + ".build")
    try:
        build._nvcc()
    except RuntimeError:
        pytest.skip("needs the CUDA toolchain")
    assert os.path.getsize(build_device_ops(str(tmp_path))) > 0


# ---- GPU: the sm_100a build vs the references and the host build ---------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", OP_NAMES)
def test_device_matches_reference_on_edges(device_ops, name):
    recs = edge_records(name)
    in_, aux = pack(recs)
    assert_matches(name, recs, device_ops(name, in_, aux), expected(name, recs))


@pytest.mark.gpu
@pytest.mark.parametrize("name", OP_NAMES)
def test_device_matches_host_build_on_random(device_ops, host_ops, name):
    in_, aux = random_records(name, N_PERM_GPU if name in SLOW_OPS else N_RANDOM_GPU, seed=2)
    got, want = device_ops(name, in_, aux), host_ops(name, in_, aux)
    if (got != want).any():
        recs = unpack(in_, aux)
        assert_matches(name, recs, got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", OP_NAMES)
def test_block_size_does_not_change_results(device_ops, name):
    """block sizes 1 and 33 do not divide the 256 table vectors load_reduce_tab copies; results stay byte-identical"""
    in_, aux = pack(edge_records(name))
    r_in, r_aux = random_records(name, 64 if name in SLOW_OPS else 4096, seed=3)
    in_, aux = np.concatenate([in_, r_in]), np.concatenate([aux, r_aux])
    ref = device_ops(name, in_, aux, block=256)
    for block in (1, 33):
        assert device_ops(name, in_, aux, block=block).tobytes() == ref.tobytes(), (name, block)
