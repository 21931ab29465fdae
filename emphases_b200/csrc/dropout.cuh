// Dropout randomness shared by every kernel that drops (sm_100a).
//
// Philox4x32-10 (Salmon et al., SC'11; the generator family torch uses):
// key = the 64-bit seed of one training forward, counter = (element index / 4
// as two words, site, 0).  One call yields the four 32-bit draws of four
// consecutive element indices; element i keeps its value iff draw[i % 4] >=
// round(p * 2^32), and kept values are scaled by 1 / (1 - p).  The counter is a
// function of the element's coordinates only (never of the thread or grid), so
// emph_dropout_keep reproduces every mask the kernels apply, and the backward
// regenerates the forward's masks from the seed instead of storing them.
//
// Element index per site (see EMPH_DROPOUT_SITE in include/emphases_b200.h):
//   row-wise sites:  packed_row * channels + channel
//   attention:       packed_query_row << 16 | key index within the sequence
//   conv blocks:     (n * width + w) * channels + channel (EMPH_DROPOUT_CONV):
//                    the position in the reference's padded tensor, item or
//                    segment n = row_seq[r], column w = r - row_start[n], so the
//                    native step (which skips rows no word reaches) and the
//                    per-kernel path draw the same mask
#pragma once

#include <stdint.h>

namespace emph {

struct Dropout {
    unsigned long long seed;
    uint32_t site;
    unsigned long long threshold;   // round(p * 2^32): 0 keeps everything
    float scale;                    // 1 / (1 - p); 1 at p = 0, 0 at p = 1
};

inline Dropout make_dropout(unsigned long long seed, uint32_t site, float p) {
    Dropout d;
    d.seed = seed;
    d.site = site;
    const double scaled = (double)p * 4294967296.0;
    d.threshold = p <= 0.f ? 0ull : (unsigned long long)(scaled + 0.5);
    d.scale = p <= 0.f ? 1.f : (p >= 1.f ? 0.f : (float)(1.0 / (1.0 - (double)p)));
    return d;
}

// the four draws of element indices 4 * group .. 4 * group + 3
__device__ __forceinline__ uint4 philox_draws(
    unsigned long long seed, uint32_t site, unsigned long long group) {
    uint32_t c0 = (uint32_t)group, c1 = (uint32_t)(group >> 32), c2 = site, c3 = 0u;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int round = 0; round < 10; ++round) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

__device__ __forceinline__ uint32_t draw_of(uint4 draws, unsigned long long index) {
    const uint32_t i = (uint32_t)index & 3u;
    return i == 0 ? draws.x : i == 1 ? draws.y : i == 2 ? draws.z : draws.w;
}

__device__ __forceinline__ bool dropout_keep(
    const Dropout& d, uint32_t site, unsigned long long index) {
    if (d.threshold == 0ull) return true;
    return (unsigned long long)draw_of(philox_draws(d.seed, site, index >> 2), index) >= d.threshold;
}

// keep multiplier (scale or 0) of element `index` from the draws of its group
__device__ __forceinline__ float dropout_factor(
    const Dropout& d, uint4 draws, unsigned long long index) {
    return (unsigned long long)draw_of(draws, index) >= d.threshold ? d.scale : 0.f;
}

}  // namespace emph
