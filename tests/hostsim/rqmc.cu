// Test-only: the randomised-QMC pieces of RZ_RENDER_RQMC (rz_sampler.cuh's replicate mapping, rz_device.cuh's replicate terms,
// segment arithmetic and rz_pixel_err_rqmc) compiled as HOST code, so that tests/test_rqmc_cpu.py can check them against numpy.
// The product only ever runs these functions inside its CUDA kernels.
#include <cstdint>

#include "../../rayz_b200/csrc/rz_device.cuh"

// n points: pixel gpix[k], pair pair[k], sample sample[k] -> rz_sobol_pair's coordinates xy[2k], xy[2k + 1] with `rqmc`
extern "C" void hostrqmc_pairs(uint64_t seed, int rqmc, const uint32_t *gpix, const uint32_t *pair, const uint32_t *sample, uint64_t n,
                               uint32_t *xy) {
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (uint64_t k = 0; k < n; k++) {
        const uint2 q = rz_sobol_pair(k0, k1, gpix[k], pair[k], sample[k], rqmc != 0);
        xy[2 * k] = q.x;
        xy[2 * k + 1] = q.y;
    }
}

// A pixel's paths' clamped luminance, quantised into its two replicate sums as the sky branch of rz_shade_segment adds them
// (path k belongs to replicate (offset + k) & 1).
extern "C" void hostrqmc_rep_sums(const float *rgb, uint32_t n, uint32_t offset, uint64_t *rep) {
    rep[0] = rep[1] = 0;
    for (uint32_t k = 0; k < n; k++) {
        const float r = rz_clamp_radiance(rgb[3 * k]), g = rz_clamp_radiance(rgb[3 * k + 1]), b = rz_clamp_radiance(rgb[3 * k + 2]);
        rep[(offset + k) & 1u] += rz_fixed32(rz_clamp_radiance(rz_luma(r, g, b)));
    }
}

extern "C" double hostrqmc_var_iid(const uint64_t *q, uint32_t n) { return rz_pixel_var_iid(q[0], q[1], q[2], q[3], n); }
extern "C" double hostrqmc_var_rep(const uint64_t *r, uint32_t n) { return rz_pixel_var_rep(r[0], r[1], n); }
extern "C" double hostrqmc_err(const uint64_t *q, uint32_t n, double gain) { return rz_pixel_err_rqmc(q[0], q[1], q[2], q[3], n, gain); }
extern "C" uint32_t hostrqmc_segments(uint32_t width) { return rz_rqmc_segments(width); }
extern "C" uint64_t hostrqmc_segment_of(uint32_t lp, uint32_t width) { return rz_rqmc_segment_of(lp, width); }

// Every segment's gain of n_local_px = rows x width pixels (accum [n][4], rep [n][2], counts n_px or every pixel n), summed in
// the order rz_rqmc_gain_kernel adds them: lane k takes pixels x0 + k, x0 + k + 32, then an xor tree over the 32 lanes; and the
// per-pixel gains it writes: the segment's gain for every pixel whose count is n, the others left as they were.
extern "C" void hostrqmc_gains(const uint64_t *accum, const uint64_t *rep, const uint32_t *n_px, uint32_t n, uint32_t n_local_px,
                               uint32_t width, double *gain, double *px_gain) {
    const uint32_t nseg = rz_rqmc_segments(width), rows = n_local_px / width;
    for (uint32_t seg = 0; seg < rows * nseg; seg++) {
        const uint32_t lr = seg / nseg, x0 = (seg - lr * nseg) * RZ_RQMC_SEGMENT, x1 = x0 + RZ_RQMC_SEGMENT < width ? x0 + RZ_RQMC_SEGMENT : width;
        double v_rep[32] = {}, v_iid[32] = {};
        for (uint32_t lane = 0; lane < 32; lane++)
            for (uint32_t x = x0 + lane; x < x1; x += 32u) {
                const uint32_t lp = lr * width + x, c = n_px ? n_px[lp] : n;
                const uint64_t *q = accum + (size_t)lp * 4;
                v_rep[lane] += rz_pixel_var_rep(rep[(size_t)lp * 2], rep[(size_t)lp * 2 + 1], c);
                v_iid[lane] += rz_pixel_var_iid(q[0], q[1], q[2], q[3], c);
            }
        for (int o = 16; o > 0; o >>= 1) {
            double r2[32], i2[32];
            for (int l = 0; l < 32; l++) { r2[l] = v_rep[l] + v_rep[l ^ o]; i2[l] = v_iid[l] + v_iid[l ^ o]; }
            for (int l = 0; l < 32; l++) { v_rep[l] = r2[l]; v_iid[l] = i2[l]; }
        }
        gain[seg] = rz_rqmc_gain(v_rep[0], v_iid[0]);
        for (uint32_t x = x0; x < x1; x++)
            if (!n_px || n_px[lr * width + x] == n) px_gain[lr * width + x] = gain[seg];
    }
}
