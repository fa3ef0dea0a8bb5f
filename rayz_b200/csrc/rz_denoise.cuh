// rz_denoise.cuh — the per-pixel and per-tap arithmetic of the edge-avoiding à-trous denoiser (rz_denoise.cu,
// rayz_cuda_denoise in include/rayz_cuda.h).  RZ_HD so that tests/hostsim/denoise.cu compiles the same FP32 code as host
// code and the CPU tests compare it with the numpy f64 restatement in tests/test_denoise_cpu.py.
//
// The filter (SVGF's spatial filter, Schied et al. 2017, on the à-trous wavelet of Dammertz et al. 2010), per pixel p:
//   Y(x) = 0.2126 x.r + 0.7152 x.g + 0.0722 x.b;  c_p: resolved linear rgb, e_p: rz_pixel_err (displayed-value error)
//   v_p  = 4 e_p^2 max(Y(c_p), 1e-4)             variance of the pixel mean's luminance (the inverse of rz_pixel_err)
//   i_p  = c_p / max(albedo_p, 1e-3),  v_p /= max(Y(albedo_p), 1e-3)^2            (demodulation)
//   g_p  = central differences of the guide depth z, indices clamped at the frame edges: ((z[x+1] - z[x-1]) / 2, ...)
//   level k, step s = 2^k, taps q = p + s (dx, dy), dx, dy in -2..2 inside the frame, h = (1, 4, 6, 4, 1) / 16:
//     gv_p = 3 x 3 binomial (1, 2, 1) blur of v around p (taps outside the frame skipped, weights renormalised)
//     w    = h[dx] h[dy] w_l w_n w_z  (rz_denoise_weight)
//     i'_p = sum w i_q / sum w,   v'_p = sum w^2 v_q / (sum w)^2   (a tap whose f32 w^2 is 0 adds nothing to the variance)
//   out_p = i_p max(albedo_p, 1e-3)                                                 (remodulation)
#pragma once
#include "rz_device.cuh"

// rz_launch_denoise's arguments (rz_denoise.cu), filled by rayz_cuda_denoise (rz_context.cu)
struct RzDenoiseArgs {
    float4 *linear;          // in: the resolved frame; out: the denoised frame (a = 1)
    uint8_t *rgb8;           // out: trunc(255 clamp(sqrt(x))) of the denoised frame
    const float *err;        // rz_pixel_err per pixel
    const float4 *albedo;    // guide albedo (rgb) + coverage
    const float4 *normal;    // guide normal (xyz) + depth (w)
    float4 *work;            // 2 x pixels: the ping-pong buffers of (demodulated rgb, variance)
    float2 *grad;            // depth gradient per pixel
    uint32_t width, height, iterations;
    float sigma_l, sigma_n, sigma_z;
};

#define RZ_DENOISE_ALBEDO_FLOOR 1e-3f
#define RZ_DENOISE_LUM_EPS 1e-4f
#define RZ_DENOISE_DEPTH_EPS 1e-2f

RZ_HD float rz_denoise_luma(float r, float g, float b) { return fmaf(0.0722f, b, fmaf(0.7152f, g, 0.2126f * r)); }

// Edge-stopping weight of tap q for pixel p, without the kernel's h[dx] h[dy]:
//   w_l = exp(-|Y(i_p) - Y(i_q)| / (sigma_l sqrt(gv_p) + 1e-4))                      (1 when gv_p = +inf)
//   w_n = clamp(n_p.n_q / (|n_p| |n_q|), 0, 1)^sigma_n if both normals are nonzero, 1 if both are zero (sky), else 0
//   w_z = exp(-|z_p - z_q| / (sigma_z |g_p . (q - p)| + 1e-2))
// yp, yq: Y of the demodulated colours; np, nq: the guide normals (xyz, mean of unit normals) with the depth in w; (ox, oy) = q - p
// in pixels.
RZ_HD float rz_denoise_weight(float yp, float yq, float gv_p, float4 np, float4 nq, float2 gp, float ox, float oy, float sigma_l,
                              float sigma_n, float sigma_z) {
    const float wl = expf(-fabsf(yp - yq) / fmaf(sigma_l, sqrtf(gv_p), RZ_DENOISE_LUM_EPS));
    const float pp = fmaf(np.x, np.x, fmaf(np.y, np.y, np.z * np.z)), qq = fmaf(nq.x, nq.x, fmaf(nq.y, nq.y, nq.z * nq.z));
    float wn;
    if (pp > 0.f && qq > 0.f) {
        const float c = fmaf(np.x, nq.x, fmaf(np.y, nq.y, np.z * nq.z)) / sqrtf(pp * qq);
        wn = powf(fminf(fmaxf(c, 0.f), 1.f), sigma_n);
    } else {
        wn = (pp > 0.f) == (qq > 0.f) ? 1.f : 0.f;
    }
    const float wz = expf(-fabsf(np.w - nq.w) / fmaf(sigma_z, fabsf(fmaf(gp.x, ox, gp.y * oy)), RZ_DENOISE_DEPTH_EPS));
    return wl * wn * wz;
}

// Demodulated colour and variance (i_p, v_p) of a pixel from its resolved colour c, error e and guide albedo a.
RZ_HD float4 rz_denoise_demodulate(float4 c, float e, float4 a) {
    const float v = 4.f * e * e * fmaxf(rz_denoise_luma(c.x, c.y, c.z), RZ_DENOISE_LUM_EPS);
    const float ya = fmaxf(rz_denoise_luma(a.x, a.y, a.z), RZ_DENOISE_ALBEDO_FLOOR);
    return make_float4(c.x / fmaxf(a.x, RZ_DENOISE_ALBEDO_FLOOR), c.y / fmaxf(a.y, RZ_DENOISE_ALBEDO_FLOOR), c.z / fmaxf(a.z, RZ_DENOISE_ALBEDO_FLOOR),
                       v / (ya * ya));
}

// Remodulated output colour (a = 1) of a filtered demodulated colour i and the guide albedo a.
RZ_HD float4 rz_denoise_remodulate(float4 i, float4 a) {
    return make_float4(i.x * fmaxf(a.x, RZ_DENOISE_ALBEDO_FLOOR), i.y * fmaxf(a.y, RZ_DENOISE_ALBEDO_FLOOR), i.z * fmaxf(a.z, RZ_DENOISE_ALBEDO_FLOOR), 1.f);
}
