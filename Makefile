# Convenience wrapper; the authoritative recipe is codex-storage-proofs-circuits_b200/build.py (what __graft_entry__.build() runs).
PKG := codex-storage-proofs-circuits_b200
NVCC ?= nvcc
NVCCFLAGS := -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -shared -ldl

all: lib cli oracle

lib: $(PKG)/libcodexcommit.so
$(PKG)/libcodexcommit.so: $(PKG)/csrc/capi.cu $(PKG)/csrc/kernels.cuh $(PKG)/csrc/poseidon2.cuh $(PKG)/csrc/fr.cuh $(PKG)/csrc/poseidon2_rc.cuh $(PKG)/csrc/fr_reduce_tab.cuh $(PKG)/csrc/capi_multi.cuh $(PKG)/csrc/slot_image.h include/codex_commit.h
	$(NVCC) $(NVCCFLAGS) -o $@ $<

cli: $(PKG)/cli
$(PKG)/cli: $(PKG)/host/cli.cpp $(PKG)/host/proof_input.cpp $(PKG)/host/proof_input.hpp $(PKG)/libcodexcommit.so
	g++ -O2 -std=c++17 -Wall -Wextra -o $@ $(PKG)/host/proof_input.cpp $(PKG)/host/cli.cpp -L$(PKG) -lcodexcommit -Wl,-rpath,'$$ORIGIN'

oracle:
	$(MAKE) -C oracle

test:
	python -m pytest tests -x -q -m "not gpu"

clean:
	rm -f $(PKG)/libcodexcommit.so $(PKG)/cli
	$(MAKE) -C oracle clean
.PHONY: all lib cli oracle test clean
