"""codex-storage-proofs-circuits_b200 -- B200 (sm_100a) slot-commitment backend for Codex storage proofs.

The package holds only what the hot path needs:
  csrc/          hand-written CUDA (BN254 Fr, Poseidon2, cell sponge, Merkle levels, path gather) + the C ABI,
                 including the NCCL communicator, sharded-slot, batched-slot and dataset entry points
  host/          C++ mirror of reference/nim/proof_input (same proc names, arguments, error behaviour) and its cli
  nim/           the Nim binding and the patched reference modules (cannot be compiled here: no Nim toolchain)
  capi.py        ctypes binding of libcodexcommit.so (include/codex_commit.h)
  sharded.py     communicator bootstrap for torch.distributed jobs + Python twins of the range planners
  dataset.py     benchmark dataset description (size distribution, per-slot seeds) + Python twin of the LPT packing
  build.py       nvcc recipe (in-tree libcodexcommit.so)

The directory name is not a Python identifier; import it with
    importlib.import_module("codex-storage-proofs-circuits_b200")
(tests/conftest.py and bench.py do exactly that).
"""
from . import capi  # noqa: F401
from .capi import CodexCommitError, Comm, Context, Dataset, Slot, SlotBuilder, load_library  # noqa: F401

__all__ = ["capi", "Context", "Slot", "SlotBuilder", "Comm", "Dataset", "CodexCommitError", "load_library"]
