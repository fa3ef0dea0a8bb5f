// Test-only: the noise estimate of progressive rendering (rz_device.cuh: rz_clamp_radiance, rz_fixed32, rz_luma_sq,
// rz_pixel_err) compiled as HOST code, so that the CPU tests can check it against numpy f64 (tests/test_progressive_cpu.py).
// The product only ever runs these functions inside its CUDA kernels.
#include <cstdint>

#include "../../rayz_b200/csrc/rz_device.cuh"

// A pixel's n path radiances rgb[n][3] quantised into its four accumulator slots as the sky branch of rz_shade_segment adds
// them (q[4]), and rz_pixel_err of such slots.
extern "C" void hostnoise_moments(const float *rgb, uint32_t n, uint64_t *q) {
    q[0] = q[1] = q[2] = q[3] = 0;
    for (uint32_t k = 0; k < n; k++) {
        const float r = rz_clamp_radiance(rgb[3 * k]), g = rz_clamp_radiance(rgb[3 * k + 1]), b = rz_clamp_radiance(rgb[3 * k + 2]);
        q[0] += rz_fixed32(r); q[1] += rz_fixed32(g); q[2] += rz_fixed32(b);
        q[3] += rz_fixed32(rz_luma_sq(r, g, b));
    }
}
extern "C" double hostnoise_pixel_err(const uint64_t *q, uint32_t n) { return rz_pixel_err(q[0], q[1], q[2], q[3], n); }
