// Philox4x32-10 (Salmon et al., SC'11; Random123), shared by the keyed per-object streams: gp_object_noise uses the
// counters (q, 0, 0, 0), gp_sample_points' permutation the counters (R, round, 1, 0).  The key is (lo32, hi32) of the
// object's int64 key, so one key per object can feed both streams.
#pragma once
#include <stdint.h>

namespace gp {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += W0;
        k1 += W1;
    }
    return c;
}

}  // namespace gp
