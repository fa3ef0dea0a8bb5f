// Test-only: the estimator of RZ_RENDER_ADAPTIVE_POOLED (rz_device.cuh's rz_pixel_u, rz_pool_u, rz_pixel_err_pooled and the
// pooled forms of rz_pixel_err_of) compiled as HOST code, so that tests/test_adaptive_pooled_cpu.py can check it against numpy.
// The product only ever runs these functions inside its CUDA kernels.
#include <cstdint>

#include "../../rayz_b200/csrc/rz_device.cuh"

extern "C" double hostpool_nu0(void) { return RZ_POOL_NU0; }
extern "C" double hostpool_u(const uint64_t *q, uint32_t n) { return rz_pixel_u(q[0], q[1], q[2], q[3], n); }
extern "C" double hostpool_err(const uint64_t *q, uint32_t n, double pool_u) { return rz_pixel_err_pooled(q[0], q[1], q[2], q[3], n, pool_u); }
extern "C" double hostpool_err_rqmc(const uint64_t *q, uint32_t n, double pool_u, double gain) {
    return rz_pixel_err_pooled_rqmc(q[0], q[1], q[2], q[3], n, pool_u, gain);
}

// Every segment's U_S of n_local_px = rows x width pixels (accum [n][4], counts n_px or every pixel n), summed in the order
// rz_segment_kernel adds them: lane k takes pixels x0 + k, x0 + k + 32, then an xor tree over the 32 lanes; the per-pixel
// copies it writes (the segment's U_S for every pixel whose count is n, the others left as they were); and every pixel's error
// as the consumers read it, rz_pixel_err_of with the per-pixel priors and, if gain is not null, per-pixel gains.
extern "C" void hostpool_pass(const uint64_t *accum, const uint32_t *n_px, uint32_t n, uint32_t n_local_px, uint32_t width,
                              const double *gain, double *pool, double *px_pool, double *err) {
    const uint32_t nseg = rz_rqmc_segments(width), rows = n_local_px / width;
    for (uint32_t seg = 0; seg < rows * nseg; seg++) {
        const uint32_t lr = seg / nseg, x0 = (seg - lr * nseg) * RZ_RQMC_SEGMENT, x1 = x0 + RZ_RQMC_SEGMENT < width ? x0 + RZ_RQMC_SEGMENT : width;
        double du[32] = {}, dd[32] = {};
        for (uint32_t lane = 0; lane < 32; lane++)
            for (uint32_t x = x0 + lane; x < x1; x += 32u) {
                const uint32_t lp = lr * width + x, c = n_px ? n_px[lp] : n;
                const uint64_t *q = accum + (size_t)lp * 4;
                if (c < 2u) continue;
                const double d = (double)(c - 1u);
                du[lane] += d * rz_pixel_u(q[0], q[1], q[2], q[3], c);
                dd[lane] += d;
            }
        for (int o = 16; o > 0; o >>= 1) {
            double a2[32], b2[32];
            for (int l = 0; l < 32; l++) { a2[l] = du[l] + du[l ^ o]; b2[l] = dd[l] + dd[l ^ o]; }
            for (int l = 0; l < 32; l++) { du[l] = a2[l]; dd[l] = b2[l]; }
        }
        pool[seg] = rz_pool_u(du[0], dd[0]);
        for (uint32_t x = x0; x < x1; x++)
            if (!n_px || n_px[lr * width + x] == n) px_pool[lr * width + x] = pool[seg];
    }
    for (uint32_t lp = 0; lp < n_local_px; lp++) err[lp] = rz_pixel_err_of((const unsigned long long *)accum + (size_t)lp * 4, n_px ? n_px[lp] : n, gain, px_pool, lp);
}
