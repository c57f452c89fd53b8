// Philox4x64-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11), with the round
// structure and constants of Random123 -- the generator numpy ships as np.random.Philox.  A counter-based generator:
// the block is a pure function of (counter, key), so every (episode, step, agent) draws its exploration uniforms on its
// own, in any launch, on any device, without a state to carry or a buffer to fill.
#pragma once

namespace marl {

constexpr unsigned long long kPhiloxM0 = 0xD2E7470EE14C6C93ULL;   // round multipliers
constexpr unsigned long long kPhiloxM1 = 0xCA5A826395121157ULL;
constexpr unsigned long long kPhiloxW0 = 0x9E3779B97F4A7C15ULL;   // key increments (golden ratio, sqrt(3) - 1)
constexpr unsigned long long kPhiloxW1 = 0xBB67AE8584CAA73BULL;

// The four output words of counter c under key (k0, k1).
__device__ __forceinline__ void philox4x64_10(unsigned long long c[4], unsigned long long k0, unsigned long long k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r > 0) { k0 += kPhiloxW0; k1 += kPhiloxW1; }
        const unsigned long long hi0 = __umul64hi(kPhiloxM0, c[0]), lo0 = kPhiloxM0 * c[0];
        const unsigned long long hi1 = __umul64hi(kPhiloxM1, c[2]), lo1 = kPhiloxM1 * c[2];
        const unsigned long long c1 = c[1], c3 = c[3];
        c[0] = hi1 ^ c1 ^ k0; c[1] = lo1; c[2] = hi0 ^ c3 ^ k1; c[3] = lo0;
    }
}

// numpy's Generator.random() conversion: the top 53 bits of the word, times 2^-53 (exact, in [0, 1)).
__device__ __forceinline__ double philox_to_unit(unsigned long long w) { return (double)(w >> 11) * 0x1.0p-53; }

// The exploration pair of agent n of episode `episode` at step `step`: key (seed, 0), counter (episode, step, n, 0);
// word 0 gives explore_u, word 1 choice_u (include/marl_b200.h, marl_act_philox).
__device__ __forceinline__ void philox_act_uniforms(unsigned long long seed, unsigned long long episode, int step, int n,
                                                    double& explore_u, double& choice_u) {
    unsigned long long c[4] = {episode, (unsigned long long)(unsigned)step, (unsigned long long)(unsigned)n, 0ULL};
    philox4x64_10(c, seed, 0ULL);
    explore_u = philox_to_unit(c[0]);
    choice_u = philox_to_unit(c[1]);
}

}  // namespace marl
