// Philox4x32-10 (Salmon et al. 2011, as defined by Random123): the counter-based generator behind the bootstrap sampler
// (parsimony.cu) and the stochastic mapping of event_mapping.cu.  oracle/ref_bootstrap.py::philox4x32_10 is the same function.
#pragma once
#include <stdint.h>

namespace bppgpu {

// c <- Philox4x32-10(c) under key (k0, k1)
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t x0 = hi1 ^ c[1] ^ k0, x2 = hi0 ^ c[3] ^ k1;
    c[0] = x0;
    c[1] = lo1;
    c[2] = x2;
    c[3] = lo0;
  }
}

}  // namespace bppgpu
