// TEST ONLY: the fr_ops.cuh dispatcher as an sm_100a kernel, one record per thread (tests/test_fr_device.py).
#include <cuda_runtime.h>

#include "fr_ops.cuh"

using namespace cdx;

__global__ void k_fr_ops(uint32_t op, const Fr* __restrict__ in, const uint32_t* __restrict__ aux, Fr* __restrict__ out,
                         uint64_t n) {
  load_reduce_tab();   // every thread of the CTA takes part in the copy, so the bounds check comes after it
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) test::fr_op(op, in + 3 * i, aux[i], out + 3 * i);
}

// in, out: n records of three Fr (device pointers); aux: n words.  Returns the launch error; *sync_err gets the error
// of the device synchronize that follows.
extern "C" int fr_ops_launch(uint32_t op, const void* in, const void* aux, void* out, uint64_t n, uint32_t block,
                             int* sync_err) {
  const uint64_t grid = (n + block - 1) / block;
  k_fr_ops<<<(unsigned)grid, block>>>(op, (const Fr*)in, (const uint32_t*)aux, (Fr*)out, n);
  const int launch_err = (int)cudaGetLastError();
  *sync_err = (int)cudaDeviceSynchronize();
  return launch_err;
}
