// Device random numbers shared by the Metropolis-Hastings kernels (mcmc.cu, emulate.cu, darcy_mh.cu).
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
// uniform in (0, 1) from 53 bits of a Philox output pair.  The top value 2^53 - 1 + 1/2 rounds to 2^53 in double: the fmin
// keeps it below 1, and every other value is (n + 1/2) / 2^53 as rounded.
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
    return fmin(((double)((((unsigned long long)hi << 32) | lo) >> 11) + 0.5) * (1.0 / 9007199254740992.0),
                1.0 - 1.0 / 9007199254740992.0);
}

// Philox4x32-10 keyed by `seed` at the counter (it, c, j, tag): the Box-Muller pair, normals 2 j and 2 j + 1 of chain c at
// step it, into *z0 and (unless z1 is NULL, when p is odd) *z1.  `tag` keeps the streams of different samplers apart.
__device__ __forceinline__ void philox_normal_pair(unsigned long long seed, int it, int c, int j, uint32_t tag, double* z0,
                                                   double* z1) {
    uint32_t ctr[4] = {(uint32_t)it, (uint32_t)c, (uint32_t)j, tag};
    philox4(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double u1 = u53(ctr[0], ctr[1]), u2 = u53(ctr[2], ctr[3]);
    const double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    *z0 = rad * cs;
    if (z1) *z1 = rad * sn;
}
// xi of the ensemble noise sqrt(2h / n_C) (U - ubar) xi (J x J; row s: source particle, column j: target particle), the one
// definition of its elements: Philox4x32-10 keyed by the seed at the counter (j >> 1, TAG_ENS, s, step), whose Box-Muller
// pair is (xi[s, 2 m], xi[s, 2 m + 1]) for m = j >> 1 -- the cosine for even j, the sine for odd j.  Word 1 carries the
// tag where fill_normal has the high half of its pair index, so the two streams never share a counter at the same
// (seed, step).  Drawn by fill_ensemble_noise_kernel (ensemble.cu) and inside the single-CTA kernels (small.cu).
constexpr uint32_t TAG_ENS = 0x454E;
__device__ __forceinline__ double2 ensemble_noise_pair(unsigned long long seed, unsigned long long step,
                                                       unsigned long long s, unsigned long long m) {
    uint32_t c[4] = {(uint32_t)m, TAG_ENS, (uint32_t)s, (uint32_t)step};
    philox4(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double rad = sqrt(-2.0 * log(u53(c[0], c[1])));
    double sn, cs;
    sincospi(2.0 * u53(c[2], c[3]), &sn, &cs);
    return make_double2(rad * cs, rad * sn);
}

// the accept test's uniform of chain c at step it: its own counter (it, c, 0xffffffff, tag)
__device__ __forceinline__ double philox_accept_uniform(unsigned long long seed, int it, int c, uint32_t tag) {
    uint32_t ctr[4] = {(uint32_t)it, (uint32_t)c, 0xffffffffu, tag};
    philox4(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
    return u53(ctr[0], ctr[1]);
}

// The random numbers of one proposal of chain c at step it, for the samplers that step all chains in lockstep
// (emulate.cu, darcy_mh.cu): z[q * zstride] ~ N(0, 1) for q < p, and the accept test's uniform as the return value.
// With mt != nullptr the chain consumes numpy's stream (mt: 624 key words, position, has_gauss; *cached: the cached
// variate) in the order np.random.normal(0, 1, p) then np.random.uniform() draw, and the advanced state is written back.
// Otherwise the normals and the uniform come from philox_normal_pair and philox_accept_uniform.
__device__ inline double mh_chain_draw(int p, int it, int c, uint32_t* mt, double* cached, unsigned long long seed,
                                       uint32_t tag, double* z, int zstride) {
    if (mt) {
        Mt rng;
        rng.key = mt; rng.pos = (int)mt[624]; rng.has_gauss = (int)mt[625]; rng.gauss = cached[0];
        for (int q = 0; q < p; ++q) z[(size_t)q * zstride] = mt_gauss(rng);
        const double u = mt_double(rng);
        mt[624] = (uint32_t)rng.pos; mt[625] = (uint32_t)rng.has_gauss; cached[0] = rng.gauss;
        return u;
    }
    for (int q2 = 0; 2 * q2 < p; ++q2) {
        philox_normal_pair(seed, it, c, q2, tag, &z[(size_t)(2 * q2) * zstride],
                           2 * q2 + 1 < p ? &z[(size_t)(2 * q2 + 1) * zstride] : nullptr);
    }
    return philox_accept_uniform(seed, it, c, tag);
}

}  // namespace ces
