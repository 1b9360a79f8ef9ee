"""nvcc recipe for libcodexcommit.so (sm_100a only, built in-tree so it travels with the repo snapshot)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcodexcommit.so")
SOURCES = ["capi.cu"]
HEADERS = ["fr.cuh", "fr_reduce_tab.cuh", "poseidon2.cuh", "poseidon2_rc.cuh", "kernels.cuh", "capi_multi.cuh", "slot_image.h", "slot_builder.h",os.path.join("..", "..", "include", "codex_commit.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "-shared", "-ldl"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB


HOST = os.path.join(HERE, "host")
CLI = os.path.join(HERE, "cli")
HOST_SOURCES = ["proof_input.cpp", "cli.cpp"]
HOST_HEADERS = ["proof_input.hpp"]


def build_host(force: bool = False) -> str:
    """g++ build of the host-side mirror of reference/nim/proof_input and its `cli`, linked against the in-tree
    libcodexcommit.so (rpath $ORIGIN, so the pair travels together)."""
    build_library()
    deps = [os.path.join(HOST, f) for f in HOST_SOURCES + HOST_HEADERS] + [LIB]
    if not force and os.path.exists(CLI) and all(os.path.getmtime(d) <= os.path.getmtime(CLI) for d in deps):
        return CLI
    cxx = shutil.which("g++") or "g++"
    cmd = [cxx, "-O2", "-std=c++17", "-Wall", "-Wextra", "-o", CLI] + [os.path.join(HOST, s) for s in HOST_SOURCES] + \
          ["-L" + HERE, "-lcodexcommit", "-Wl,-rpath,$ORIGIN"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("g++ failed:\n" + res.stdout + res.stderr)
    return CLI


def ensure_built() -> None:
    """Build the CUDA library / host cli only if the artefact is MISSING (fresh checkout on a box with nvcc); an existing
    build is never replaced behind the caller's back.  This is not a fallback: it produces the same sm_100a library."""
    if not os.path.exists(LIB):
        build_library(force=True)
    if not os.path.exists(CLI):
        build_host(force=True)


if __name__ == "__main__":
    import sys
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_host(force="--force" in sys.argv))
