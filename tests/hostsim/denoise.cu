// Test-only: the denoiser's per-pixel and per-tap arithmetic (rz_denoise.cuh: rz_denoise_weight, rz_denoise_demodulate,
// rz_denoise_remodulate) compiled as HOST code, so that the CPU tests can check it against numpy f64 (tests/test_denoise_cpu.py).
// The product only ever runs these functions inside its CUDA kernels.
#include <cstdint>

#include "../../rayz_b200/csrc/rz_denoise.cuh"

// n weights: per tap, t[11 k ..] = yp, yq, gv_p, np.xyzw, nq.xyzw; o[4 k ..] = g_p.xy, q - p; s = sigma_l, sigma_n, sigma_z
extern "C" void hostdenoise_weights(const float *t, const float *o, const float *s, uint32_t n, float *out) {
    for (uint32_t k = 0; k < n; k++) {
        const float *a = t + 11 * (size_t)k;
        out[k] = rz_denoise_weight(a[0], a[1], a[2], make_float4(a[3], a[4], a[5], a[6]), make_float4(a[7], a[8], a[9], a[10]),
                                   make_float2(o[4 * (size_t)k], o[4 * (size_t)k + 1]), o[4 * (size_t)k + 2], o[4 * (size_t)k + 3], s[0], s[1], s[2]);
    }
}
// n pixels: c[4k..], e[k], a[4k..] -> (i, v)[4k..] and the remodulated i
extern "C" void hostdenoise_demodulate(const float *c, const float *e, const float *a, uint32_t n, float *iv, float *remod) {
    for (uint32_t k = 0; k < n; k++) {
        const float4 al = make_float4(a[4 * k], a[4 * k + 1], a[4 * k + 2], a[4 * k + 3]);
        const float4 r = rz_denoise_demodulate(make_float4(c[4 * k], c[4 * k + 1], c[4 * k + 2], c[4 * k + 3]), e[k], al);
        const float4 m = rz_denoise_remodulate(r, al);
        iv[4 * k] = r.x; iv[4 * k + 1] = r.y; iv[4 * k + 2] = r.z; iv[4 * k + 3] = r.w;
        remod[4 * k] = m.x; remod[4 * k + 1] = m.y; remod[4 * k + 2] = m.z; remod[4 * k + 3] = m.w;
    }
}
