// Philox4x32-10 addressed variates — device twin of oracle/gpo_rng.h (same address scheme, DESIGN.md "RNG addressing").
//   counter = (idx', stream, purpose, sweep), key = (seed_lo, seed_hi)
//   uniform(idx): counter idx,     first 64 output bits -> (x>>11 + 0.5) * 2^-53  in (0,1)
//   normal(idx) : counter idx>>1,  Box-Muller on (u1,u2): even idx -> r cos(2 pi u2), odd idx -> r sin(2 pi u2)
#pragma once
#include <cstdint>

namespace gpirt {

enum Purpose : uint32_t {
    P_INIT_F_Z = 0, P_INIT_BETA = 1, P_ESS_Z = 2, P_ESS_U = 3, P_FSTAR_Z = 4, P_THETA_U = 5, P_BETA_Z = 6, P_BETA_U = 7,
    P_PPC_U = 8   // posterior predictive replicates (opts.ppc): drawn outside the chain, which never reads them
};

// sweep_dev (optional): device word added to `sweep` at run time — lets a CUDA graph of a whole sweep be replayed with a
// new sweep counter (a one-thread kernel inside the graph bumps the word) without touching kernel parameters.
struct RngKey { uint32_t k0, k1, sweep; const uint32_t* sweep_dev; };
__device__ __forceinline__ uint32_t rng_sweep(const RngKey& key) { return key.sweep_dev ? key.sweep + *key.sweep_dev : key.sweep; }

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3,
                                                       uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
#ifdef __CUDA_ARCH__
        uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0, hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
#else
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += W0; k1 += W1;
    }
}

__host__ __device__ __forceinline__ double u01_from_bits(uint32_t lo, uint32_t hi) {
    uint64_t x = ((uint64_t)hi << 32) | lo;
    return ((double)(x >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ double rng_uniform(const RngKey& key, uint32_t purpose, uint32_t stream, uint32_t idx) {
    uint32_t c0 = idx, c1 = stream, c2 = purpose, c3 = rng_sweep(key);
    philox4x32_10(c0, c1, c2, c3, key.k0, key.k1);
    return u01_from_bits(c0, c1);
}

// both members of the Box-Muller pair with counter `pair` (elements 2*pair and 2*pair+1 of the stream)
__device__ __forceinline__ void rng_normal_pair(const RngKey& key, uint32_t purpose, uint32_t stream, uint32_t pair,
                                                double& z_even, double& z_odd) {
    uint32_t c0 = pair, c1 = stream, c2 = purpose, c3 = rng_sweep(key);
    philox4x32_10(c0, c1, c2, c3, key.k0, key.k1);
    double u1 = u01_from_bits(c0, c1), u2 = u01_from_bits(c2, c3);
    double r = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    z_even = r * c;
    z_odd = r * s;
}

__device__ __forceinline__ double rng_normal(const RngKey& key, uint32_t purpose, uint32_t stream, uint32_t idx) {
    double a, b;
    rng_normal_pair(key, purpose, stream, idx >> 1, a, b);
    return (idx & 1u) ? b : a;
}

} // namespace gpirt
