// rz_misc.cu — K5 resolve/quantise and K6 FP32 peak microbenchmark.
#include <cuda_runtime.h>
#include <stdint.h>

// ---------------------------------------------------------------------------------------------
// K5.  Fixed-point accumulators -> linear float4 + gamma-2 RGB8.
// Restates `acc_color.div(spp)` (renderer.zig:94-95: multiply by the reciprocal) and writePPM's
// per-pixel transform (image.zig:35-38): V3.sqrt (x > 0 ? sqrt(x) : 0, vec.zig:87-93) ->
// clamp(0,1) -> u8 = trunc(x * 255).  Done in f64 like the reference so that the truncation
// lands on the same side; W*H threads, negligible next to the path kernel.
// Output rows may live on ANOTHER GPU (peer pointers): with out_row_stride/out_row_offset the
// kernel scatters this device's compact band-interleaved rows straight into the gather root's
// full-shard buffers over NVLink, i.e. resolve and gather are one kernel.
// The same kernel writes the per-pixel noise estimate (out_err: rz_pixel_err of the four slots) when asked.
// ---------------------------------------------------------------------------------------------
#include "rz_device.cuh"   // rz_pixel_err

struct RzResolveArgs {
    const unsigned long long *accum;  // [n_local_px][4]
    float4 *out_linear;               // nullable
    uint8_t *out_rgb8;                // nullable
    float *out_err;                   // nullable: displayed-value standard error per pixel (needs slot 3, RZ_RENDER_MOMENTS)
    uint32_t n_local_px, width;
    uint32_t spp;                     // samples summed in the accumulators (cumulative over RZ_RENDER_ACCUMULATE batches)
    // local row lr of this device -> destination row ((lr / band) * dev_count + dev_index) * band + lr % band
    uint32_t dev_index, dev_count, band_rows;
};

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
    if (a.out_err) a.out_err[dst] = (float)rz_pixel_err(q0.x, q0.y, q1, a.accum[(size_t)lp * 4 + 3], a.spp);
    const double inv = 1.0 / (double)a.spp;
    const double s = 2.3283064365386962890625e-10;  // 2^-32
    const double r = (double)q0.x * s * inv, g = (double)q0.y * s * inv, b = (double)q1 * s * inv;
    if (a.out_linear) a.out_linear[dst] = make_float4((float)r, (float)g, (float)b, 1.0f);
    if (a.out_rgb8) {
        const double sr = r > 0 ? sqrt(r) : 0, sg = g > 0 ? sqrt(g) : 0, sb = b > 0 ? sqrt(b) : 0;
        const double cr = fmin(fmax(sr, 0.0), 1.0), cg = fmin(fmax(sg, 0.0), 1.0), cb = fmin(fmax(sb, 0.0), 1.0);
        a.out_rgb8[dst * 3 + 0] = (uint8_t)(cr * 255.0);
        a.out_rgb8[dst * 3 + 1] = (uint8_t)(cg * 255.0);
        a.out_rgb8[dst * 3 + 2] = (uint8_t)(cb * 255.0);
    }
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
#define RZ_NOISE_GRID 256
struct RzNoisePartial { double sum, sum2, max; unsigned long long above; };

__global__ void __launch_bounds__(256) rz_noise_reduce_kernel(const unsigned long long *__restrict__ accum, uint32_t n_local_px, uint32_t n,
                                                              double target, RzNoisePartial *__restrict__ out) {
    __shared__ double s_sum[256], s_sum2[256], s_max[256];
    __shared__ unsigned long long s_above[256];
    double sum = 0, sum2 = 0, mx = 0;
    unsigned long long above = 0;
    for (uint32_t lp = blockIdx.x * 256u + threadIdx.x; lp < n_local_px; lp += RZ_NOISE_GRID * 256u) {
        const unsigned long long *q = accum + (size_t)lp * 4;
        const double e = (double)(float)rz_pixel_err(q[0], q[1], q[2], q[3], n);   // the value out_err shows
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

extern "C" uint32_t rz_noise_grid(void) { return RZ_NOISE_GRID; }
// out: RZ_NOISE_GRID x 4 words (sum, sum2, max as doubles, then the count as an integer)
extern "C" cudaError_t rz_launch_noise_reduce(const unsigned long long *accum, uint32_t n_local_px, uint32_t n, double target, void *out,
                                              cudaStream_t stream) {
    rz_noise_reduce_kernel<<<RZ_NOISE_GRID, 256, 0, stream>>>(accum, n_local_px, n, target, (RzNoisePartial *)out);
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
