// fr_ops.cuh -- TEST ONLY.  One dispatcher over the field and Poseidon2 operations of fr.cuh / poseidon2.cuh on RAW
// limb values (no conversion in or out), so tests/test_fr_device.py can pin each lazily reduced result bit for bit
// against a big-integer reference.  Compiled twice: by nvcc for sm_100a (fr_ops.cu, the inline-PTX primitives) and by
// g++ with -DCDX_HOST_EMUL (fr_ops_host.cpp, the C emulation in tests/host_emul/fr_rows_host.h).
#pragma once
#include "../../codex-storage-proofs-circuits_b200/csrc/poseidon2.cuh"

namespace cdx {
namespace test {

// op numbers; tests/test_fr_device.py keeps the same list in OPS
enum FrOp : uint32_t {
  OP_MONT_MUL = 0,      // out0 = mont_mul(in0, in1)
  OP_MONT_SQR,          // out0 = mont_sqr(in0)
  OP_REDUCE_TAB,        // out0 = reduce_tab(in0, aux)          aux = carry, 0 or 1
  OP_ADD_REDUCE,        // out0 = add_reduce(in0, in1)
  OP_REDUCE_ONCE,       // out0 = reduce_once(in0)
  OP_ADD_MOD,           // out0 = add_mod(in0, in1)
  OP_DBL_MOD,           // out0 = dbl_mod(in0)
  OP_TO_MONT,           // out0 = to_mont(in0)
  OP_FROM_MONT,         // out0 = from_mont(in0)
  OP_MONT_FROM_U32,     // out0 = mont_from_u32(aux)
  OP_SBOX,              // out0 = sbox(in0)
  OP_MIX_EXTERNAL,      // out0..2 = mix_external(in0, in1, in2)
  OP_MIX_INTERNAL,      // out0..2 = mix_internal(in0, in1, in2)
  OP_ABSORB,            // out0 = absorb(in0, in1)
  OP_ABSORB_ONE,        // out0 = absorb_one(in0)
  OP_SPONGE_IV,         // out0 = sponge_iv(aux)                aux = rate
  OP_PERMUTE,           // out0..2 = permute(in0, in1, in2)
  OP_COMPRESS_KEYED,    // out0 = compress_keyed(in0, in1, aux) aux = key
  OP_COUNT
};

// in: three words and the auxiliary word of one record; out: three words (the ones an op does not produce are zero)
CDX_D void fr_op(uint32_t op, const Fr* in, uint32_t aux, Fr* out) {
  Fr x = in[0], y = in[1], z = in[2];
  Fr r = fr_zero();
  switch (op) {
    case OP_MONT_MUL: r = mont_mul(x, y); break;
    case OP_MONT_SQR: r = mont_sqr(x); break;
    case OP_REDUCE_TAB: r = reduce_tab(x, aux); break;
    case OP_ADD_REDUCE: r = add_reduce(x, y); break;
    case OP_REDUCE_ONCE: r = reduce_once(x); break;
    case OP_ADD_MOD: r = add_mod(x, y); break;
    case OP_DBL_MOD: r = dbl_mod(x); break;
    case OP_TO_MONT: r = to_mont(x); break;
    case OP_FROM_MONT: r = from_mont(x); break;
    case OP_MONT_FROM_U32: r = mont_from_u32(aux); break;
    case OP_SBOX: r = sbox(x); break;
    case OP_MIX_EXTERNAL: mix_external(x, y, z); out[0] = x; out[1] = y; out[2] = z; return;
    case OP_MIX_INTERNAL: mix_internal(x, y, z); out[0] = x; out[1] = y; out[2] = z; return;
    case OP_ABSORB: r = absorb(x, y); break;
    case OP_ABSORB_ONE: r = absorb_one(x); break;
    case OP_SPONGE_IV: r = sponge_iv((int)aux); break;
    case OP_PERMUTE: permute(x, y, z); out[0] = x; out[1] = y; out[2] = z; return;
    case OP_COMPRESS_KEYED: r = compress_keyed(x, y, aux); break;
    default: break;
  }
  out[0] = r;
  out[1] = out[2] = fr_zero();
}

}  // namespace test
}  // namespace cdx
