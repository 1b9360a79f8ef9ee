// TEST ONLY: the fr_ops.cuh dispatcher built with g++ against the C emulation of the PTX primitives
// (tests/host_emul/fr_rows_host.h), one record after the other (tests/test_fr_device.py).
#define CDX_HOST_EMUL 1
#include "fr_ops.cuh"

using namespace cdx;

// in, out: n records of three Fr; aux: n words
extern "C" void fr_ops_host(uint32_t op, const Fr* in, const uint32_t* aux, Fr* out, uint64_t n) {
  for (uint64_t i = 0; i < n; ++i) test::fr_op(op, in + 3 * i, aux[i], out + 3 * i);
}
