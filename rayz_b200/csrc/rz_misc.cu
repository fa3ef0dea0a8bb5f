// rz_misc.cu — K5 resolve/quantise and K6 FP32 peak microbenchmark.

// ---------------------------------------------------------------------------------------------
// K5.  Fixed-point accumulators -> linear float4 + gamma-2 RGB8.
// Restates `acc_color.div(spp)` (renderer.zig:94-95: multiply by the reciprocal) and writePPM's
// per-pixel transform (image.zig:35-38): V3.sqrt (x > 0 ? sqrt(x) : 0, vec.zig:87-93) ->
// clamp(0,1) -> u8 = trunc(x * 255).  Done in f64 like the reference so that the truncation
// lands on the same side; W*H threads, negligible next to the path kernel.
// Output rows may live on ANOTHER GPU (peer pointers): with out_row_stride/out_row_offset the
// kernel scatters this device's compact band-interleaved rows straight into the gather root's
// full-shard buffers over NVLink, i.e. resolve and gather are one kernel.
// The same kernel writes the per-pixel noise estimate (out_err: rz_pixel_err of the four slots) and the pixels' sample counts
// (out_spp) when asked.  An adaptive frame divides each pixel by its own count (n_px), in the same f64 arithmetic: a pixel
// with c samples resolves exactly as the same pixel of a uniform c-spp render.
// ---------------------------------------------------------------------------------------------
#include "rz_device.cuh"   // rz_pixel_err, rz_quantise_rgb8
#include "rz_launch.h"     // RzResolveArgs, RzNoisePartial

__global__ void __launch_bounds__(256) rz_resolve_kernel(const RzResolveArgs a) {
    const uint32_t lp = blockIdx.x * blockDim.x + threadIdx.x;
    if (lp >= a.n_local_px) return;
    const ulonglong2 q0 = *reinterpret_cast<const ulonglong2 *>(a.accum + (size_t)lp * 4);
    const unsigned long long q1 = a.accum[(size_t)lp * 4 + 2];
    size_t dst = lp;
    if (a.dev_count > 1u) {
        const uint32_t lr = lp / a.width, i = lp - lr * a.width;
        const uint32_t lb = lr / a.band_rows, within = lr - lb * a.band_rows;
        dst = (size_t)((lb * a.dev_count + a.dev_index) * a.band_rows + within) * a.width + i;
    }
    const uint32_t n = a.n_px ? a.n_px[lp] : a.spp;
    if (a.out_spp) a.out_spp[dst] = n;
    if (a.out_err) {
        const unsigned long long q3 = a.accum[(size_t)lp * 4 + 3];
        a.out_err[dst] = (float)(a.gain ? rz_pixel_err_rqmc(q0.x, q0.y, q1, q3, n, a.gain[lp]) : rz_pixel_err(q0.x, q0.y, q1, q3, n));
    }
    const double inv = 1.0 / (double)n;
    const double s = 2.3283064365386962890625e-10;  // 2^-32
    const double r = (double)q0.x * s * inv, g = (double)q0.y * s * inv, b = (double)q1 * s * inv;
    if (a.out_linear) a.out_linear[dst] = make_float4((float)r, (float)g, (float)b, 1.0f);
    if (a.out_rgb8) rz_quantise_rgb8(r, g, b, a.out_rgb8, dst);
}

extern "C" cudaError_t rz_launch_resolve(const RzResolveArgs *a, cudaStream_t stream) {
    if (a->n_local_px == 0) return cudaSuccess;
    rz_resolve_kernel<<<(a->n_local_px + 255) / 256, 256, 0, stream>>>(*a);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Frame summary of the noise estimate: per CTA of a FIXED grid (RZ_NOISE_GRID x 256), sum of e, sum of e^2, max e and the
// count of pixels with e > target over the pixels lp = cta * 256 + tid + k * grid * 256, reduced in a fixed tree.  The host
// adds the CTAs' partials in order: no floating-point atomics, so two identical calls give identical summaries.
// ---------------------------------------------------------------------------------------------

// n_px (nullable): per-pixel sample counts of an adaptive frame, else every pixel has n samples.  gain (nullable): RZ_RENDER_RQMC's
// per-pixel gains.
__global__ void __launch_bounds__(256) rz_noise_reduce_kernel(const unsigned long long *__restrict__ accum, const uint32_t *__restrict__ n_px,
                                                              const double *__restrict__ gain, uint32_t n_local_px, uint32_t n, double target, RzNoisePartial *__restrict__ out) {
    __shared__ double s_sum[256], s_sum2[256], s_max[256];
    __shared__ unsigned long long s_above[256];
    double sum = 0, sum2 = 0, mx = 0;
    unsigned long long above = 0;
    for (uint32_t lp = blockIdx.x * 256u + threadIdx.x; lp < n_local_px; lp += RZ_NOISE_GRID * 256u) {
        const unsigned long long *q = accum + (size_t)lp * 4;
        const double e = (double)(float)rz_pixel_err_of(q, n_px ? n_px[lp] : n, gain, lp);   // the value out_err shows
        sum += e; sum2 += e * e; mx = fmax(mx, e); above += e > target ? 1u : 0u;
    }
    s_sum[threadIdx.x] = sum; s_sum2[threadIdx.x] = sum2; s_max[threadIdx.x] = mx; s_above[threadIdx.x] = above;
    __syncthreads();
    for (uint32_t h = 128; h > 0; h >>= 1) {
        if (threadIdx.x < h) {
            s_sum[threadIdx.x] += s_sum[threadIdx.x + h]; s_sum2[threadIdx.x] += s_sum2[threadIdx.x + h];
            s_max[threadIdx.x] = fmax(s_max[threadIdx.x], s_max[threadIdx.x + h]); s_above[threadIdx.x] += s_above[threadIdx.x + h];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = RzNoisePartial{s_sum[0], s_sum2[0], s_max[0], s_above[0]};
}

extern "C" cudaError_t rz_launch_noise_reduce(const unsigned long long *accum, const uint32_t *n_px, const double *gain,
                                              uint32_t n_local_px, uint32_t n, double target, RzNoisePartial *out, cudaStream_t stream) {
    rz_noise_reduce_kernel<<<RZ_NOISE_GRID, 256, 0, stream>>>(accum, n_px, gain, n_local_px, n, target, out);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// RZ_RENDER_RQMC: the gain G of every segment of the device's local rows (rz_rqmc_gain of the segment's sums of V_rep and V_iid),
// into seg_gain[row][rz_rqmc_segments(width)], and into px_gain[lp] for every pixel whose count is n, the frame's largest: every
// pixel of a uniform frame; of an adaptive one, the pixels the next stopping test reads.  A pixel that stopped keeps the gain its
// test read, so its error stays what the test saw while its segment's other pixels take more samples.  One warp per segment:
// lane k adds its pixels x0 + k, x0 + k + 32 in that order, then a fixed xor tree that leaves the sums in every lane; no
// floating-point atomics, so the gain is a function of the segment's sums only, wherever the row renders.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) rz_rqmc_gain_kernel(const unsigned long long *__restrict__ accum, const unsigned long long *__restrict__ rep,
                                                           const uint32_t *__restrict__ n_px, uint32_t n, uint32_t n_local_px, uint32_t width,
                                                           double *__restrict__ seg_gain, double *__restrict__ px_gain) {
    const uint32_t nseg = rz_rqmc_segments(width), rows = n_local_px / width;
    const uint32_t seg = blockIdx.x * 4u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
    if (seg >= rows * nseg) return;   // the whole warp
    const uint32_t lr = seg / nseg, x0 = (seg - lr * nseg) * RZ_RQMC_SEGMENT, x1 = min(x0 + RZ_RQMC_SEGMENT, width);
    double v_rep = 0.0, v_iid = 0.0;
    for (uint32_t x = x0 + lane; x < x1; x += 32u) {
        const uint32_t lp = lr * width + x, c = n_px ? n_px[lp] : n;
        const unsigned long long *q = accum + (size_t)lp * 4;
        v_rep += rz_pixel_var_rep(rep[(size_t)lp * 2], rep[(size_t)lp * 2 + 1], c);
        v_iid += rz_pixel_var_iid(q[0], q[1], q[2], q[3], c);
    }
    for (int o = 16; o > 0; o >>= 1) {
        v_rep += __shfl_xor_sync(0xffffffffu, v_rep, o);
        v_iid += __shfl_xor_sync(0xffffffffu, v_iid, o);
    }
    const double g = rz_rqmc_gain(v_rep, v_iid);
    if (lane == 0) seg_gain[seg] = g;
    for (uint32_t x = x0 + lane; x < x1; x += 32u) {
        const uint32_t lp = lr * width + x;
        if (!n_px || n_px[lp] == n) px_gain[lp] = g;
    }
}

// Doubles of the segment-gain buffer for n_local_px pixels in rows of `width` (px_gain: n_local_px doubles).
extern "C" size_t rz_rqmc_gain_words(uint32_t n_local_px, uint32_t width) { return width ? (size_t)(n_local_px / width) * rz_rqmc_segments(width) : 0; }
extern "C" cudaError_t rz_launch_rqmc_gain(const unsigned long long *accum, const unsigned long long *rep, const uint32_t *n_px, uint32_t n,
                                           uint32_t n_local_px, uint32_t width, double *seg_gain, double *px_gain, cudaStream_t stream) {
    const size_t segs = rz_rqmc_gain_words(n_local_px, width);
    if (segs == 0) return cudaSuccess;
    rz_rqmc_gain_kernel<<<(unsigned)((segs + 3) / 4), 128, 0, stream>>>(accum, rep, n_px, n, n_local_px, width, seg_gain, px_gain);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// K6.  FP32 peak: 16 independent FFMA chains per thread, 3-register form (no immediates), all
// SMs, 8 CTAs x 256 threads per SM.  flops = 2 * FFMAs.  This is the measured roofline
// denominator for the path kernel (MEASURED_PEAKS.json carries no FP32 figure).
// ---------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) rz_ffma_peak_kernel(float *sink, float a, float b, int iters) {
    float x[16];
#pragma unroll
    for (int i = 0; i < 16; i++) x[i] = (float)(threadIdx.x + i) * 1e-3f;
    if (MODE == 0) {
        // x = x*a + b : 16 independent chains, scalar multiplier/addend
#pragma unroll 1
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int u = 0; u < 8; u++) {
#pragma unroll
                for (int i = 0; i < 16; i++) x[i] = fmaf(x[i], a, b);
            }
        }
    } else if (MODE == 2) {
        // packed FP32x2 (fma.rn.f32x2 -> SASS FFMA2): 8 chains of float2 = the same 16 FMAs per step
        float2 p[8];
#pragma unroll
        for (int i = 0; i < 8; i++) p[i] = make_float2(x[2 * i], x[2 * i + 1]);
        const float2 a2 = make_float2(a, a), b2 = make_float2(b, b);
#pragma unroll 1
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int u = 0; u < 8; u++) {
#pragma unroll
                for (int i = 0; i < 8; i++) p[i] = __ffma2_rn(p[i], a2, b2);
            }
        }
#pragma unroll
        for (int i = 0; i < 8; i++) { x[2 * i] = p[i].x; x[2 * i + 1] = p[i].y; }
    } else {
        // acc[i][j] += y[i]*z[j] : SGEMM-like outer product, three distinct registers per FFMA
        float y[4], z[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { y[i] = a + (float)(threadIdx.x & 3) * 1e-6f * (float)(i + 1); z[i] = b * (float)(i + 1) + (float)(threadIdx.x & 7) * 1e-7f; }
#pragma unroll 1
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int u = 0; u < 8; u++) {
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) x[i * 4 + j] = fmaf(y[i], z[j], x[i * 4 + j]);
            }
            // keep y/z loop-variant without adding FP work to the count (1 op per 128 FFMAs)
            y[0] = -y[0];
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; i++) s += x[i];
    if (s == 123.456f) sink[0] = s;  // never true; keeps the chains alive
}

// FFMAs per thread per `iters` unit = 8 * 16 = 128
extern "C" cudaError_t rz_launch_ffma_peak(float *sink, int grid, int iters, int mode, cudaStream_t stream) {
    if (mode == 0) rz_ffma_peak_kernel<0><<<grid, 256, 0, stream>>>(sink, 0.999f, 1e-3f, iters);
    else if (mode == 2) rz_ffma_peak_kernel<2><<<grid, 256, 0, stream>>>(sink, 0.999f, 1e-3f, iters);
    else rz_ffma_peak_kernel<1><<<grid, 256, 0, stream>>>(sink, 0.999f, 1e-3f, iters);
    return cudaGetLastError();
}
