// Philox4x32-10 counter-based generator (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; the
// constants and round function of Random123's philox4x32_10).  __host__ __device__ so that the host mirror used by
// zl_sample_uniform and the kernel in sample.cu are the same code.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ZL_HD __host__ __device__ __forceinline__
#else
#define ZL_HD inline
#endif

namespace zl {

ZL_HD void philox4x32_10(const uint32_t ctr_in[4], const uint32_t key_in[2], uint32_t out[4]) {
    uint32_t c0 = ctr_in[0], c1 = ctr_in[1], c2 = ctr_in[2], c3 = ctr_in[3];
    uint32_t k0 = key_in[0], k1 = key_in[1];
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        const uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0;
    out[1] = c1;
    out[2] = c2;
    out[3] = c3;
}

// the sampling draw: key = the task's 64-bit seed, counter = {draw_index, 0, 0, 0}; u = ((w0 >> 8) + 1) * 2^-24 in (0, 1]
ZL_HD float sample_uniform(uint64_t seed, uint32_t draw_index) {
    const uint32_t ctr[4] = {draw_index, 0u, 0u, 0u};
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    uint32_t w[4];
    philox4x32_10(ctr, key, w);
    return (float)((w[0] >> 8) + 1u) * (1.0f / 16777216.0f);
}

}  // namespace zl
