"""The C-ABI library loads and exports every symbol include/codex_commit.h declares (no compute calls: CPU only)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def header_functions():
    src = open(os.path.join(ROOT, "include", "codex_commit.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(cdx_[a-z0-9_]+)\s*\(", src)))


def test_header_and_binding_agree(pkg):
    names = header_functions()
    assert len(names) >= 30
    assert sorted(pkg.capi.SYMBOLS) == names


def test_library_exports_every_declared_symbol(pkg):
    lib = ctypes.CDLL(pkg.capi.LIB_PATH)
    for name in header_functions():
        assert getattr(lib, name) is not None, name
    assert pkg.load_library().cdx_abi_version() == 2


def test_pure_host_helpers(pkg):
    lib = pkg.load_library()
    # layer arithmetic of merkleTreeWorker (merkle/bn254.nim:29-60)
    assert lib.cdx_merkle_total_nodes(1, 1) == 2 and lib.cdx_merkle_num_layers(1, 1) == 2
    assert lib.cdx_merkle_total_nodes(1, 0) == 1 and lib.cdx_merkle_num_layers(1, 0) == 1
    assert lib.cdx_merkle_total_nodes(5, 1) == 5 + 3 + 2 + 1 and lib.cdx_merkle_num_layers(5, 1) == 4
    assert lib.cdx_merkle_total_nodes(64, 1) == 127
    assert lib.cdx_status_string(-3).decode().startswith("number of cells")


def test_no_device_is_a_loud_error(pkg):
    """Without a GPU the context cannot be created -- there is no CPU fallback behind the ABI."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(pkg.CodexCommitError) as e:
        pkg.Context(0)
    assert e.value.status == pkg.capi.CDX_ERR_CUDA


def test_product_never_touches_the_oracle():
    """the product path may not import, link, call or execute anything under oracle/"""
    pkgdir = os.path.join(ROOT, "codex-storage-proofs-circuits_b200")
    pat = re.compile(r"(from|import)\s+\.*oracle|oracle/|codex_oracle|coracle|pyoracle")
    for dp, _, files in os.walk(pkgdir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                text = open(os.path.join(dp, f), errors="ignore").read()
                assert not pat.search(text), f"{os.path.join(dp, f)} references the oracle"


def test_header_is_plain_c(tmp_path):
    """cgo / Nim importc / ctypes-style consumers compile include/codex_commit.h as C: no C++ in the declarations"""
    import subprocess
    hdr = os.path.join(ROOT, "include")
    src = tmp_path / "use.c"
    src.write_text('#include "codex_commit.h"\n'
                   "int probe(cdx_ctx* c, cdx_slot* s, unsigned char* out) {\n"
                   "  unsigned long long idx[1] = {0};\n"
                   "  if (cdx_slot_root(s, out) != CDX_OK) return 1;\n"
                   "  return cdx_slot_cell_paths(s, (const uint64_t*)idx, 1, 32, out, 0) + (c == 0);\n"
                   "}\n")
    for cc, std in (("gcc", "-std=c99"), ("g++", "-std=c++11")):
        res = subprocess.run([cc, std, "-Wall", "-Werror", "-pedantic", "-x", "c" if cc == "gcc" else "c++", "-I", hdr, "-c", str(src), "-o",
                              str(tmp_path / "use.o")], capture_output=True, text=True)
        assert res.returncode == 0, res.stderr


def test_planners_and_comm_without_a_gpu(pkg):
    """host-only entry points of the multi-GPU half of the ABI: the range planners need no device; a one-rank communicator
    needs a context (so a GPU), and asking for several ranks without NCCL's id is an argument error, not a crash"""
    t, ranges = pkg.capi.plan_block_ranges(1638400, 8)
    assert t == 13 and ranges[7] == (7 * 204800, 204800)
    t, ranges = pkg.capi.plan_block_ranges(3, 4)                       # fewer chunks than ranks: empty shards
    assert t == 0 and sorted(c for _, c in ranges) == [0, 1, 1, 1]
    assert pkg.capi.block_ranges_top_level(1 << 20, [(0, 1 << 19), (1 << 19, 1 << 19)]) == 19
    lib = pkg.load_library()
    assert lib.cdx_comm_rank(None) == 0 and lib.cdx_comm_size(None) == 1
    assert lib.cdx_group_size(None) == 0 and lib.cdx_dataset_kept_slot(None) is None


def test_nim_binding_declares_every_symbol():
    """the Nim delivery (cannot be compiled here: no Nim toolchain) at least covers the whole ABI: the generated binding has
    one importc per header function, and regenerating it changes nothing"""
    import subprocess
    import sys
    path = os.path.join(ROOT, "codex-storage-proofs-circuits_b200", "nim", "codexcommit_abi.nim")
    before = open(path).read()
    declared = set(re.findall(r"^proc (cdx_[a-z0-9_]+)\*\(", before, flags=re.M))
    assert declared == set(header_functions())
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_nim_binding.py")], check=True, capture_output=True)
    assert open(path).read() == before


def build_c_example(tmp_path):
    import subprocess
    pkg_dir = os.path.join(ROOT, "codex-storage-proofs-circuits_b200")
    exe = str(tmp_path / "commit_dataset")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-O1", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "commit_dataset.c"), "-L" + pkg_dir, "-lcodexcommit", "-Wl,-rpath," + pkg_dir, "-o", exe], check=True)
    return exe


def test_plain_c_example_links_and_fails_loudly_without_a_gpu(pkg, tmp_path):
    """examples/commit_dataset.c: the ABI is usable from a C99 compiler (no C++ in the header, every symbol links); without
    a device the program reports that there is no CPU path"""
    import subprocess
    import torch
    exe = build_c_example(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present: the GPU suite runs the example")
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert res.returncode == 2 and "no CPU path" in res.stderr
