// Test-only: the low-discrepancy sampler (rz_sampler.cuh, RZ_RENDER_SOBOL) compiled as HOST code, so that the CPU tests can
// check it against an independent numpy restatement and test its stratification (tests/test_sampler_cpu.py).  The product only
// ever runs these functions inside its CUDA kernels.
#include <cstdint>

#include "../../rayz_b200/csrc/rz_device.cuh"

// n points: pixel gpix[k], pair pair[k], sample sample[k] -> the 32-bit coordinates xy[2k], xy[2k + 1] and the pair's base seed
extern "C" void hostsampler_pairs(uint64_t seed, const uint32_t *gpix, const uint32_t *pair, const uint32_t *sample, uint64_t n,
                                  uint32_t *xy, uint32_t *base) {
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (uint64_t k = 0; k < n; k++) {
        const uint2 q = rz_sobol_pair(k0, k1, gpix[k], pair[k], sample[k]);
        xy[2 * k] = q.x;
        xy[2 * k + 1] = q.y;
        base[k] = rz_sobol_pair_seed(k0, k1, gpix[k], pair[k]);
    }
}

// The uniforms the kernels use: camera jitter (x, y), lens (radius, angle), time, then u.x, u.y of bounces 1..depth.
extern "C" void hostsampler_uniforms(uint64_t seed, uint32_t gpix, uint32_t sample, uint32_t depth, float *u) {
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const float2 j = rz_sobol_u01(k0, k1, gpix, RZ_PAIR_CAMERA_JITTER, sample), l = rz_sobol_u01(k0, k1, gpix, RZ_PAIR_CAMERA_LENS, sample);
    u[0] = j.x; u[1] = j.y; u[2] = l.x; u[3] = l.y; u[4] = rz_sobol_u01(k0, k1, gpix, RZ_PAIR_CAMERA_TIME, sample).x;
    for (uint32_t s = 1; s <= depth; s++) {
        const float2 b = rz_sobol_u01(k0, k1, gpix, rz_pair_bounce(s), sample);
        u[3 + 2 * s] = b.x; u[4 + 2 * s] = b.y;
    }
}
