// rz_denoise.cu — edge-avoiding à-trous denoiser of the accumulated frame (rayz_cuda_denoise, include/rayz_cuda.h).
// Runs on the gather root alone, over whole-frame buffers in image order: the resolve kernel has put the linear frame and the
// per-pixel error there, rz_guides_kernel the albedo, normal and depth.  The formulas are in rz_denoise.cuh.
//   rz_denoise_prepare_kernel : demodulate (i, v) into the first ping-pong buffer, the depth gradient into its own
//   rz_atrous_kernel          : one level (step 2^k) of the 5 x 5 à-trous filter, ping-pong buffer to ping-pong buffer
//   rz_denoise_finish_kernel  : remodulate into the linear output, then writePPM's f64 quantisation of that f32 value
// One thread per pixel, 2-D blocks; every buffer is float4 (or float2) per pixel so a tap is one vector load, and the frame's
// buffers stay in the 126 MB L2 at config 2 (1200 x 675: 13 MB per float4 buffer) across the levels.
#include <cuda_runtime.h>
#include <stdint.h>

#include "rz_denoise.cuh"   // RzDenoiseArgs and the arithmetic


#define RZ_DN_BX 32
#define RZ_DN_BY 8

__global__ void __launch_bounds__(RZ_DN_BX * RZ_DN_BY) rz_denoise_prepare_kernel(const RzDenoiseArgs a) {
    const uint32_t x = blockIdx.x * RZ_DN_BX + threadIdx.x, y = blockIdx.y * RZ_DN_BY + threadIdx.y;
    if (x >= a.width || y >= a.height) return;
    const size_t p = (size_t)y * a.width + x;
    a.work[p] = rz_denoise_demodulate(a.linear[p], a.err[p], a.albedo[p]);
    const uint32_t xl = x > 0 ? x - 1 : 0, xr = x + 1 < a.width ? x + 1 : x, yu = y > 0 ? y - 1 : 0, yd = y + 1 < a.height ? y + 1 : y;
    const float zl = a.normal[(size_t)y * a.width + xl].w, zr = a.normal[(size_t)y * a.width + xr].w;
    const float zu = a.normal[(size_t)yu * a.width + x].w, zd = a.normal[(size_t)yd * a.width + x].w;
    a.grad[p] = make_float2(0.5f * (zr - zl), 0.5f * (zd - zu));
}

__global__ void __launch_bounds__(RZ_DN_BX * RZ_DN_BY) rz_atrous_kernel(const RzDenoiseArgs a, const float4 *__restrict__ in,
                                                                         float4 *__restrict__ out, int step) {
    const int x = (int)(blockIdx.x * RZ_DN_BX + threadIdx.x), y = (int)(blockIdx.y * RZ_DN_BY + threadIdx.y);
    const int W = (int)a.width, H = (int)a.height;
    if (x >= W || y >= H) return;
    const size_t p = (size_t)y * W + x;
    const float4 cp = in[p], np = a.normal[p];
    const float2 gp = a.grad[p];
    // 3 x 3 binomial blur of the variance around p
    float gv = 0.f, gk = 0.f;
#pragma unroll
    for (int dy = -1; dy <= 1; dy++) {
#pragma unroll
        for (int dx = -1; dx <= 1; dx++) {
            const int qx = x + dx, qy = y + dy;
            if (qx < 0 || qx >= W || qy < 0 || qy >= H) continue;
            const float k = (float)((2 - dx * dx) * (2 - dy * dy));
            gv = fmaf(k, in[(size_t)qy * W + qx].w, gv);
            gk += k;
        }
    }
    gv /= gk;
    const float yp = rz_denoise_luma(cp.x, cp.y, cp.z);
    const float h[5] = {1.f / 16.f, 4.f / 16.f, 6.f / 16.f, 4.f / 16.f, 1.f / 16.f};
    float sw = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, sv = 0.f;
#pragma unroll 1
    for (int dy = -2; dy <= 2; dy++) {
        const int qy = y + dy * step;
        if (qy < 0 || qy >= H) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; dx++) {
            const int qx = x + dx * step;
            if (qx < 0 || qx >= W) continue;
            const size_t q = (size_t)qy * W + qx;
            const float4 cq = in[q];
            const float w = h[dx + 2] * h[dy + 2] *
                            rz_denoise_weight(yp, rz_denoise_luma(cq.x, cq.y, cq.z), gv, np, a.normal[q], gp, (float)(dx * step),
                                              (float)(dy * step), a.sigma_l, a.sigma_n, a.sigma_z);
            sw += w;
            sr = fmaf(w, cq.x, sr); sg = fmaf(w, cq.y, sg); sb = fmaf(w, cq.z, sb);
            const float w2 = w * w;
            if (w2 > 0.f) sv = fmaf(w2, cq.w, sv);
        }
    }
    // sum w > 0: the centre tap's w_l and w_z are 1 and its w_n is 1 up to rounding
    const float inv = 1.f / sw;
    out[p] = make_float4(sr * inv, sg * inv, sb * inv, sv * inv * inv);
}

__global__ void __launch_bounds__(RZ_DN_BX * RZ_DN_BY) rz_denoise_finish_kernel(const RzDenoiseArgs a, const float4 *__restrict__ in) {
    const uint32_t x = blockIdx.x * RZ_DN_BX + threadIdx.x, y = blockIdx.y * RZ_DN_BY + threadIdx.y;
    if (x >= a.width || y >= a.height) return;
    const size_t p = (size_t)y * a.width + x;
    const float4 o = rz_denoise_remodulate(in[p], a.albedo[p]);
    a.linear[p] = o;
    rz_quantise_rgb8((double)o.x, (double)o.y, (double)o.z, a.rgb8, p);
}

// prepare -> iterations x à-trous -> finish on one stream; iterations >= 1
extern "C" cudaError_t rz_launch_denoise(const RzDenoiseArgs *a, cudaStream_t stream) {
    const dim3 block(RZ_DN_BX, RZ_DN_BY), grid((a->width + RZ_DN_BX - 1) / RZ_DN_BX, (a->height + RZ_DN_BY - 1) / RZ_DN_BY);
    const size_t npx = (size_t)a->width * a->height;
    rz_denoise_prepare_kernel<<<grid, block, 0, stream>>>(*a);
    for (uint32_t k = 0; k < a->iterations; k++)
        rz_atrous_kernel<<<grid, block, 0, stream>>>(*a, a->work + (k & 1u) * npx, a->work + ((k + 1u) & 1u) * npx, 1 << k);
    rz_denoise_finish_kernel<<<grid, block, 0, stream>>>(*a, a->work + (a->iterations & 1u) * npx);
    return cudaGetLastError();
}
