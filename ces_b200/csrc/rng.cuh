// Device random numbers shared by the Metropolis-Hastings kernels (mcmc.cu, emulate.cu).
//
// Mt restates numpy's legacy RandomState on the MT19937 state of the caller's global generator (624 words, position,
// cached Gaussian): next_double = (a >> 5, b >> 6) / 2^53, the polar Box-Muller of legacy_gauss with its cached second
// variate.  A chain that draws from it consumes exactly the variates np.random.normal / np.random.uniform would have
// produced and leaves the state where they would have left it.  Every other chain uses Philox4x32-10 keyed by the
// caller's seed, with a counter the caller builds from (iteration, chain, index).
#pragma once
#include <cstdint>

namespace ces {

struct Mt {
    uint32_t* key;
    int pos;
    int has_gauss;
    double gauss;
};

__device__ inline void mt_twist(uint32_t* mt) {
    const uint32_t UP = 0x80000000u, LO = 0x7fffffffu, MA = 0x9908b0dfu;
    int i = 0;
    uint32_t yv;
    for (; i < 624 - 397; ++i) {
        yv = (mt[i] & UP) | (mt[i + 1] & LO);
        mt[i] = mt[i + 397] ^ (yv >> 1) ^ ((yv & 1u) ? MA : 0u);
    }
    for (; i < 623; ++i) {
        yv = (mt[i] & UP) | (mt[i + 1] & LO);
        mt[i] = mt[i + (397 - 624)] ^ (yv >> 1) ^ ((yv & 1u) ? MA : 0u);
    }
    yv = (mt[623] & UP) | (mt[0] & LO);
    mt[623] = mt[396] ^ (yv >> 1) ^ ((yv & 1u) ? MA : 0u);
}
__device__ __forceinline__ uint32_t mt_next(Mt& s) {
    if (s.pos >= 624) { mt_twist(s.key); s.pos = 0; }
    uint32_t yv = s.key[s.pos++];
    yv ^= yv >> 11;
    yv ^= (yv << 7) & 0x9d2c5680u;
    yv ^= (yv << 15) & 0xefc60000u;
    yv ^= yv >> 18;
    return yv;
}
__device__ __forceinline__ double mt_double(Mt& s) {
    const int a = (int)(mt_next(s) >> 5), b = (int)(mt_next(s) >> 6);
    return (a * 67108864.0 + b) / 9007199254740992.0;
}
__device__ inline double mt_gauss(Mt& s) {             // numpy legacy_gauss
    if (s.has_gauss) {
        const double t = s.gauss;
        s.has_gauss = 0;
        s.gauss = 0.0;
        return t;
    }
    double x1, x2, r2;
    do {
        x1 = 2.0 * mt_double(s) - 1.0;
        x2 = 2.0 * mt_double(s) - 1.0;
        r2 = x1 * x1 + x2 * x2;
    } while (r2 >= 1.0 || r2 == 0.0);
    const double f = sqrt(-2.0 * log(r2) / r2);
    s.gauss = f * x1;
    s.has_gauss = 1;
    return f * x2;
}

__device__ __forceinline__ void philox4(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}
// uniform in (0, 1) from 53 bits of a Philox output pair
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
    return ((double)((((unsigned long long)hi << 32) | lo) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}

}  // namespace ces
