// w-fsa_b200/csrc/philox.hpp -- Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011),
// the counter-based generator of path sampling (kernels_sample.cuh).  One implementation for the device and the host, so
// that wfsa_philox4x32_10 (include/wfsa_host.h) pins the bits the kernels draw.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define WFSA_HD __host__ __device__ __forceinline__
#else
#define WFSA_HD inline
#endif

namespace wfsa {

WFSA_HD void philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int i = 0; i < 10; ++i) {
        if (i) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// uniform in [0, 1) with 53 random bits: choice d of draw r of string s under key (seed & 0xffffffff, seed >> 32)
WFSA_HD double philox_uniform(uint32_t d, uint32_t r, uint32_t s, const uint32_t key[2])
{
    const uint32_t ctr[4] = {d, r, s, 0u};
    uint32_t o[4];
    philox4x32_10(ctr, key, o);
    return (double)((((uint64_t)o[0] << 32) | o[1]) >> 11) * 0x1p-53;
}

}  // namespace wfsa
