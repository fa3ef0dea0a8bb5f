// rz_launch.h — the kernel units' launch interface: every extern "C" function rz_context.cu calls, and the argument records
// that only the host and one unit share.  rz_context.cu and every unit that defines one of these functions include it, so a
// definition whose parameters drift from its declaration is a compile error (two C-linkage functions of one name) instead of
// a call that passes its arguments wrongly at run time.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct RzPathArgs; struct RzGuideArgs; struct RzMatteArgs; struct RzDenoiseArgs; struct RzBvhNode;   // rz_device.cuh, rz_denoise.cuh: by pointer only

// ------------------------------------------------------------------------------ K0 (rz_ids.cu)
struct RzRefNode { double low[3], high[3]; int32_t left, right, start, end; };   // BVH of hit.zig:101-108, children by index (RefBuilder)

struct RzIdsArgs {
    const RzRefNode *nodes;     // reference-shaped tree (host build restating hit.zig:130-161)
    const uint32_t *order;      // hittables order after the build's sorts
    const double4 *c64;         // [n] (cx,cy,cz,r)   caller's sphere order
    const double4 *v64;         // [n] (vx,vy,vz,0)
    uint32_t n_spheres, n_nodes;
    double look_from[3], px_du[3], px_dv[3], px_origin[3];
    uint32_t width, height;
    int use_bvh;
    int32_t *out;
    unsigned int *err;          // device error word: bit 2 = traversal stack overflow (never silently dropped)
};

extern "C" cudaError_t rz_launch_ids(const RzIdsArgs *a, cudaStream_t stream);

// ------------------------------------------------------------------------------ K5 resolve, noise, segment pass, K6 (rz_misc.cu)
struct RzResolveArgs {
    const unsigned long long *accum;  // [n_local_px][4]
    float4 *out_linear;               // nullable
    uint8_t *out_rgb8;                // nullable
    float *out_err;                   // nullable: displayed-value standard error per pixel (needs slot 3, RZ_RENDER_MOMENTS)
    uint32_t *out_spp;                // nullable: the pixel's sample count (rayz_cuda_pixel_samples)
    const uint32_t *n_px;             // nullable: per-pixel sample counts of an adaptive frame (rz_adaptive.cu); null: spp
    const double *gain;               // nullable: RZ_RENDER_RQMC's per-pixel gains (rz_segment_kernel); out_err is then rz_pixel_err_rqmc
    const double *pool;               // nullable: RZ_RENDER_ADAPTIVE_POOLED's per-pixel priors (rz_segment_kernel); out_err is then pooled
    uint32_t n_local_px, width;
    uint32_t spp;                     // samples summed in the accumulators (cumulative over RZ_RENDER_ACCUMULATE batches)
    // local row lr of this device -> destination row ((lr / band) * dev_count + dev_index) * band + lr % band
    uint32_t dev_index, dev_count, band_rows;
};

#define RZ_NOISE_GRID 256   // CTAs of the noise reduction's fixed grid, one RzNoisePartial each (rz_noise_reduce_kernel)
struct RzNoisePartial { double sum, sum2, max; unsigned long long above; };

extern "C" cudaError_t rz_launch_resolve(const RzResolveArgs *a, cudaStream_t stream);
extern "C" cudaError_t rz_launch_passes_resolve(const RzResolveArgs *a, const unsigned long long *passes, float4 *out, size_t plane,
                                                cudaStream_t stream);
extern "C" cudaError_t rz_launch_noise_reduce(const unsigned long long *accum, const uint32_t *n_px, const double *gain, const double *pool,
                                              uint32_t n_local_px, uint32_t n, double target, RzNoisePartial *out, cudaStream_t stream);
extern "C" size_t rz_rqmc_gain_words(uint32_t n_local_px, uint32_t width);
extern "C" cudaError_t rz_launch_rqmc_gain(const unsigned long long *accum, const unsigned long long *rep, const uint32_t *n_px, uint32_t n,
                                           uint32_t n_local_px, uint32_t width, double *seg_gain, double *px_gain, cudaStream_t stream);
extern "C" cudaError_t rz_launch_segment_pass(const unsigned long long *accum, const unsigned long long *rep, const uint32_t *n_px, uint32_t n,
                                              uint32_t n_local_px, uint32_t width, double *seg_gain, double *px_gain, double *seg_pool,
                                              double *px_pool, cudaStream_t stream);
extern "C" cudaError_t rz_launch_ffma_peak(float *sink, int grid, int iters, int mode, cudaStream_t stream);

// ------------------------------------------------------------------------------ adaptive pixel lists (rz_adaptive.cu)
extern "C" size_t rz_list_scratch_words(uint32_t n_local_px);
extern "C" size_t rz_list_count_word(uint32_t n_local_px);
extern "C" cudaError_t rz_launch_pixel_list(const unsigned long long *accum, const double *gain, const double *pool, uint32_t *n_px,
                                            uint32_t n_local_px, uint32_t n_cur, uint32_t add,
                                            float target, uint32_t *list, uint32_t *scratch, cudaStream_t stream);
extern "C" cudaError_t rz_launch_fill_u32(uint32_t *p, uint32_t n, uint32_t v, cudaStream_t stream);

// ------------------------------------------------------------------------------ K1 (rz_path.cu)
extern "C" cudaError_t rz_path_warm(void);
extern "C" size_t rz_primary_smem_bytes(const RzPathArgs *a);
extern "C" cudaError_t rz_launch_primary(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_launch_bin_lists(const RzPathArgs *a, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_second_grid(const RzPathArgs *a, int collect_stats, int sm_count, int *grid);
extern "C" cudaError_t rz_launch_second(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_launch_path(const RzPathArgs *a, int rays_per_thread, int collect_stats, int sm_count,
                                      cudaStream_t stream, int *grid_out);

// ------------------------------------------------------------------------------ the staged K1's sort (rz_sort.cu)
extern "C" size_t rz_bin_scratch_bytes(void);
extern "C" cudaError_t rz_bin_sort(const unsigned short *keys_in, const unsigned int *count, uint32_t cap, unsigned int *bins,
                                   unsigned short *keys_out, uint32_t *idx_out, uint32_t ue_max, uint32_t ue_div, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_sort_warm(void);

// ------------------------------------------------------------------------------ K2 (rz_wavefront.cu)
extern "C" cudaError_t rz_wavefront_render(const RzPathArgs *a, int sm_count, int collect_stats, cudaStream_t stream,
                                           void **scratch, size_t *scratch_bytes, uint32_t *launches);
extern "C" void rz_wavefront_free(void *scratch);

// ------------------------------------------------------------------------------ K3 and the guide buffers (rz_bvh_trace.cu)
extern "C" cudaError_t rz_bvh_warm(void);
extern "C" cudaError_t rz_launch_bvh(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_launch_bvh_stage(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_launch_guides(const RzGuideArgs *g, cudaStream_t stream);
extern "C" cudaError_t rz_launch_mattes(const RzMatteArgs *g, cudaStream_t stream);

// ------------------------------------------------------------------------------ K4 (rz_bvh_build.cu)
extern "C" size_t rz_lbvh_scratch_bytes(uint32_t n);
extern "C" cudaError_t rz_bvh_finalize(RzBvhNode *nodes, uint32_t n_nodes, cudaStream_t stream);
extern "C" cudaError_t rz_lbvh_build(uint32_t n, int leaf_max, const double4 *c64, const double4 *v64, const uint32_t *mat, void *scratch,
                                     size_t scratch_bytes, RzBvhNode *nodes, float4 *o_cr, float4 *o_vel, double4 *o_c64,
                                     double4 *o_v64, uint32_t *o_mat, int32_t *o_orig, cudaStream_t stream);

// ------------------------------------------------------------------------------ denoiser (rz_denoise.cu)
extern "C" cudaError_t rz_launch_denoise(const RzDenoiseArgs *a, cudaStream_t stream);
