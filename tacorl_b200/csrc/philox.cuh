// Counter-based Philox4x32-10 (Salmon et al., SC'11), shared by the replay sampler and the rollout policy's noise.
// oracle/replay_oracle.py restates it in numpy.
#pragma once

namespace tacorl {

struct U4 { unsigned x, y, z, w; };

__device__ __forceinline__ U4 philox4x32_10(U4 c, unsigned k0, unsigned k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c;
}

}  // namespace tacorl
