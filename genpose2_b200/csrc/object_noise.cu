// Keyed per-object initial noise of the ODE sampler (gp_object_noise): object b's block of N(0, sigma[b]^2) samples is
// a function of keys[b] and sigma[b] alone, never of b, B or the other keys (DESIGN.md section 4.6f).
//
// Philox4x32-10 (Salmon et al., SC'11; Random123) keyed with (lo32, hi32) of keys[b].  Element e = r*9 + c of the
// object's [R,9] block belongs to Box-Muller pair p = e / 2; pair p takes words 2*(p % 2), 2*(p % 2) + 1 of the
// Philox output for counter (p / 2, 0, 0, 0).  One thread makes one Philox call: pairs 2q, 2q+1, elements 4q .. 4q+3.
#include "common.cuh"

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

// u = (w + 0.5) * 2^-32 in (0, 1), float64
__device__ __forceinline__ double philox_uniform(uint32_t w) { return ((double)w + 0.5) * 0x1p-32; }

__global__ void object_noise_kernel(const int64_t *__restrict__ keys, const float *__restrict__ sigma, int B, int R,
                                    float *__restrict__ noise) {
    const int per_obj = R * 9;
    const int calls = (per_obj + 3) / 4;
    const long long q_all = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q_all >= (long long)B * calls) return;
    const int b = (int)(q_all / calls), q = (int)(q_all - (long long)b * calls);
    const uint64_t key = (uint64_t)keys[b];
    const uint4 w = philox4x32_10(make_uint4((uint32_t)q, 0u, 0u, 0u), (uint32_t)key, (uint32_t)(key >> 32));
    const float s = sigma[b];
    float *out = noise + (size_t)b * per_obj;
    const uint32_t words[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int k = 0; k < 2; ++k) {   // pair p = 2q + k
        const int e = 4 * q + 2 * k;
        if (e >= per_obj) break;
        const double rad = sqrt(-2.0 * log(philox_uniform(words[2 * k])));
        const double ang = 6.283185307179586 * philox_uniform(words[2 * k + 1]);
        out[e] = __fmul_rn((float)(rad * cos(ang)), s);
        if (e + 1 < per_obj) out[e + 1] = __fmul_rn((float)(rad * sin(ang)), s);
    }
}

}  // namespace gp

extern "C" int gp_object_noise(const int64_t *keys, const float *sigma, int B, int R, float *noise, gp_stream_t s) {
    GP_REQUIRE(B >= 1 && R >= 1, "gp_object_noise: bad sizes B=%d R=%d", B, R);
    GP_REQUIRE(R <= (1 << 26), "gp_object_noise: R=%d too large", R);
    GP_REQUIRE(keys && sigma && noise, "gp_object_noise: null pointer");
    const long long threads = (long long)B * ((R * 9 + 3) / 4);
    const int block = 256;
    gp::object_noise_kernel<<<(unsigned)((threads + block - 1) / block), block, 0, gp::as_stream(s)>>>(keys, sigma, B, R,
                                                                                                        noise);
    GP_CHECK_LAUNCH("gp_object_noise");
    return GP_OK;
}
