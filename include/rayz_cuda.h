/*
 * rayz_cuda.h — C ABI of the B200-native path-tracing backend for rayz.
 *
 * This is the drop-in boundary for ONE hot path of the reference renderer: the per-pixel
 * sample loop `Tracer.render` (reference src/renderer.zig:72-101) and everything it calls
 * (Camera.getRay camera.zig:59-90, bounceRay renderer.zig:103-126, BVH.findHit hit.zig:181-216,
 * Sphere.hitInner geom.zig:38-66, Material.scatter material.zig:73-177, and the
 * gamma/clamp/u8 step of Image.writePPM image.zig:35-38).
 *
 * The reference has no FFI today; the seam is cut at `Tracer.render()`.  A Zig host declares
 * these entry points as `extern fn` + `extern struct` (see INTEGRATION.md and zig/), copies
 * its MemPool (ecs.zig:22-27) into the flat arrays of RzScene, its Camera (camera.zig:9-16)
 * into RzCamera, calls rayz_cuda_render, and widens the float result back into `img.pixels`.
 *
 * Conventions
 *   - plain C, POD structs, little-endian, no pointers-to-pointers inside payloads;
 *   - the library OWNS all device memory; the caller owns every host array and may free it as
 *     soon as the call returns (copy semantics);
 *   - every call returns RZ_OK (0) or a negative RZ_ERR_*; rayz_cuda_last_error() gives text;
 *   - one host thread per context (the reference is single threaded, renderer.zig:80-97);
 *   - there is NO CPU fallback: without a CUDA device rayz_cuda_create fails with RZ_ERR_CUDA.
 */
#ifndef RAYZ_CUDA_H
#define RAYZ_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RAYZ_CUDA_ABI_VERSION 3

enum {
    RZ_OK = 0,
    RZ_ERR_INVALID_ARG = -1,
    RZ_ERR_CUDA = -2,
    RZ_ERR_NCCL = -3, /* reserved: peer exchange failure (P2P copy) */
    RZ_ERR_OOM = -4,
    RZ_ERR_UNSUPPORTED = -5,
    RZ_ERR_NO_SCENE = -6,
    RZ_ERR_INTERNAL = -7 /* a device-side capacity was exceeded during the render (queue slot, traversal stack): work
                          * would have been dropped, so the result is withheld instead of returned darker */
};

/* Material kinds — order of `Material = union(enum)` in material.zig:162-165. */
enum { RZ_MAT_DIFFUSE = 0, RZ_MAT_METALLIC = 1, RZ_MAT_DIELECTRIC = 2 };
/* Texture kinds — order of `Texture = union(enum)` in material.zig:41-43. */
enum { RZ_TEX_CHECKER = 0, RZ_TEX_SOLID = 1 };
/* DiffuseScatterMethod — material.zig:67-71 (default HEMISPHERE, :74). */
enum { RZ_DIFFUSE_UNIT_SPHERE = 0, RZ_DIFFUSE_UNIT_SPHERE_SURFACE = 1, RZ_DIFFUSE_HEMISPHERE = 2 };

/* Kernel variants (RzRenderParams.variant). */
enum {
    RZ_VARIANT_AUTO = 0,      /* staged K1 when the scene fits shared memory and the frame (width x height x spp)
                               * has >= 2^26 paths, else the BVH kernel (the two agree up to a pixel or two:
                               * FP32 sphere test against exact boxes)                                 */
    RZ_VARIANT_MEGA = 1,      /* K1: scene staged in shared memory; primary kernel -> sorted stages (culled
                               * brute force) -> persistent kernel for the tail of the paths: the BVH
                               * kernel, or the brute-force megakernel without a host-built tree
                               * (DESIGN.md section 3)                                             */
    RZ_VARIANT_WAVEFRONT = 2, /* K2: staged wavefront with warp-ballot compaction             */
    RZ_VARIANT_BVH = 3,       /* K3: persistent megakernel traversing the device BVH          */
    RZ_VARIANT_MEGA_SINGLE = 4 /* K1 as ONE persistent kernel (every segment brute force, paths
                               * regenerated in place): the pure FP32-bound form, 52 % of FP32 peak */
};

/*
 * Flattened MemPool (ecs.zig:22-27).  Index i of the sphere arrays is `spheres.items[i]`
 * (geom.zig:11-14: center: Ray{origin,dir}, radius, material handle); material/texture arrays
 * are indexed by Handle.idx (ecs.zig:6-17).  All reals are the reference's f64; the library
 * derives its own FP32 structure-of-arrays device layout from them.
 */
typedef struct RzScene {
    uint32_t n_spheres;
    uint32_t n_materials;
    uint32_t n_textures;
    uint32_t reserved0;
    const double *sphere_center;     /* [n_spheres][3]  Sphere.center.origin                  */
    const double *sphere_velocity;   /* [n_spheres][3]  Sphere.center.dir (0 = stationary)    */
    const double *sphere_radius;     /* [n_spheres]                                           */
    const uint32_t *sphere_material; /* [n_spheres]     MaterialHandle.idx                    */
    const uint32_t *mat_kind;        /* [n_materials]   RZ_MAT_*                              */
    const double *mat_fuzz;          /* [n_materials]   MetallicMaterial.fuzz (else 0)        */
    const double *mat_ior;           /* [n_materials]   DielectricMaterial.refractive_index   */
    const uint32_t *mat_texture;     /* [n_materials]   TextureHandle.idx (unused: dielectric)*/
    const uint32_t *mat_method;      /* [n_materials]   RZ_DIFFUSE_*; NULL => all HEMISPHERE  */
    const uint32_t *tex_kind;        /* [n_textures]    RZ_TEX_*                              */
    const double *tex_color;         /* [n_textures][3] SolidTexture.color                    */
    const double *tex_scale;         /* [n_textures]    CheckerTexture.scale                  */
    const uint32_t *tex_even;        /* [n_textures]    CheckerTexture.even handle            */
    const uint32_t *tex_odd;         /* [n_textures]    CheckerTexture.odd handle             */
} RzScene;

/* Field-for-field copy of `Camera` (camera.zig:10-16), filled by the unchanged Camera.init. */
typedef struct RzCamera {
    double look_from[3];
    double px_du[3];
    double px_dv[3];
    double px_origin[3];
    double defocus_u[3];
    double defocus_v[3];
    int32_t defocus; /* bool: defocus_angle > 0 (camera.zig:55) */
    int32_t reserved0;
} RzCamera;

/*
 * Render request.  Image rows are dealt to shards in round-robin bands:
 *   global row j belongs to shard (j / band_rows) % shard_count.
 * A context with D devices splits its own rows over its devices the same way, so a process
 * that drives shard s of S with D devices behaves as shards s*D..s*D+D-1 of S*D.
 * Results of a shard are COMPACT (its rows only, in increasing j).  shard_count <= 1 means the
 * whole image.  The random stream is keyed by the GLOBAL pixel index, sample and bounce, so
 * any sharding reproduces the full-frame render bit for bit: which kernels run (AUTO's choice, the number of sorted stages)
 * depends on the scene and the whole frame only, never on the shard, the device count or the memory that was free.
 */
typedef struct RzRenderParams {
    uint32_t width;
    uint32_t height;
    uint32_t spp;           /* Tracer.samples_per_px (renderer.zig:24)          */
    uint32_t max_depth;     /* Tracer.max_bounces   (renderer.zig:23)           */
    uint64_t seed;          /* Philox key                                        */
    uint32_t sample_offset; /* first sample index (batches: RZ_RENDER_ACCUMULATE) */
    uint32_t variant;       /* RZ_VARIANT_*                                      */
    float t_min;            /* FP32 stand-in for renderer.zig:107's 1e-10; 0 => 1e-4 */
    uint32_t shard_index;
    uint32_t shard_count;
    uint32_t band_rows;     /* 0 => 4 */
    uint32_t collect_stats; /* !=0: run the counter-instrumented kernel build    */
    uint32_t flags;         /* RZ_RENDER_* bits, 0 = defaults                    */
} RzRenderParams;

/* RzRenderParams.flags */
#define RZ_RENDER_SERIAL_PASSES 1u /* staged K1: run the passes back to back on one stream instead of
                                    * overlapping them on two, so that RzTiming.primary_ms and
                                    * kernel_ms - primary_ms are clean per-kernel durations (profiling) */
#define RZ_RENDER_MOMENTS 2u       /* also sum each path's luminance squared (Y = 0.2126 r + 0.7152 g + 0.0722 b) in the
                                    * fourth accumulator slot, so that rayz_cuda_noise can estimate the per-pixel error;
                                    * changes no pixel of the image (one more atomic per path that ends in the sky) */
#define RZ_RENDER_ACCUMULATE 4u    /* progressive rendering: add this batch to the sums of the previous render instead of
                                    * starting over, and resolve by the cumulative sample count.  Radiance is summed in
                                    * integers, so batches [0,a) + [a,b) + ... reproduce one render of all the samples bit
                                    * for bit when every batch runs the same kernel family (brute force: MEGA, MEGA_SINGLE,
                                    * WAVEFRONT; or BVH).  AUTO picks each batch's family by that batch's frame size, and the
                                    * two families agree up to a pixel or two (see RZ_VARIANT_AUTO): pin the variant where
                                    * bit equality matters.  Refused with RZ_ERR_INVALID_ARG, the sums untouched, unless the
                                    * previous render succeeded with the same width, height, shard_index/count, band_rows,
                                    * seed, max_depth, t_min, camera and RZ_RENDER_MOMENTS bit on this context, no scene
                                    * upload or differently shaped reserve came in between, sample_offset equals the previous
                                    * batch's sample_offset + spp, and the cumulative count stays below 2^32.  A render that
                                    * fails ends the accumulation.  *out_paths counts this call's paths only.  With
                                    * rayz_cuda_render_device(sync = 0), the next batch checks the previous one's device
                                    * error word before it adds to its sums. */

/* Noise summary of the accumulated frame (rayz_cuda_noise).  Errors are standard errors of the DISPLAYED value
 * (gamma 2, as writePPM shows it) in units of [0, 1]: one 8-bit step is 1/255.  +inf while samples < 2. */
typedef struct RzNoise {
    uint64_t samples;  /* samples per pixel summed so far (cumulative over RZ_RENDER_ACCUMULATE batches) */
    uint32_t n_pixels; /* pixels of the context's rows                                                   */
    uint32_t n_above;  /* pixels whose error exceeds the caller's target                                */
    double mean_err;   /* mean over the pixels                                                           */
    double rms_err;    /* root mean square over the pixels                                               */
    double max_err;
} RzNoise;

typedef struct RzConfig {
    int32_t n_devices;     /* 0 => 1 */
    int32_t device_ids[8]; /* CUDA ordinals; device_ids[0] is the gather root   */
    uint32_t flags;        /* RZ_CFG_* bits, 0 = defaults */
} RzConfig;

/* RzConfig.flags: who builds the BVH of the K3 traversal kernel at rayz_cuda_upload_scene (the
 * counterpart of bvh.build, renderer.zig:78 / hit.zig:130-161).  Default: binned-SAH on the host for
 * scenes below 8192 spheres (best tree, negligible time), LBVH on the device above. */
#define RZ_CFG_BVH_BUILD_HOST 1u   /* always the host binned-SAH builder                */
#define RZ_CFG_BVH_BUILD_DEVICE 2u /* always the device LBVH builder (rz_bvh_build.cu)  */

/* Counters of the last render with collect_stats != 0 (summed over devices). */
typedef struct RzStats {
    uint64_t paths;            /* primary samples == reference "rays" (renderer.zig:90) */
    uint64_t segments;         /* closest-hit queries == bounceRay calls with depth > 0 */
    uint64_t sphere_tests;     /* ray-sphere quadratic evaluations                       */
    uint64_t node_tests;       /* BVH box tests (BVH variants)                           */
    uint64_t hits_diffuse;
    uint64_t hits_metallic;
    uint64_t hits_dielectric;
    uint64_t ended_sky;
    uint64_t ended_absorbed;
    uint64_t ended_depth;
} RzStats;

/* Device timings of the last render call, CUDA events on the library's stream(s). */
typedef struct RzTiming {
    float kernel_ms;    /* path kernel(s) only: max over devices                    */
    float resolve_ms;   /* resolve/quantise kernel: max over devices                */
    float total_ms;     /* clear + path + resolve + peer gather (+ D2H if host API) */
    uint32_t launches;  /* kernels launched by the call, all devices                */
    uint32_t n_static;  /* stationary spheres in the device layout                  */
    uint32_t n_moving;  /* moving spheres in the device layout                      */
    uint32_t variant;   /* variant that actually ran (AUTO resolved)                */
    uint32_t bvh_build_us; /* K3 BVH build inside the last rayz_cuda_upload_scene, microseconds:
                            * host SAH wall time, or device LBVH by CUDA events (max over devices) */
    float primary_ms;      /* staged K1: sum of the primary (camera-segment) kernels' durations; a clean
                            * share of kernel_ms only with RZ_RENDER_SERIAL_PASSES (passes overlap otherwise) */
    uint32_t passes;       /* staged K1: passes (primary / sort + sorted stages / tail kernel) of the render, else 0 */
    float second_ms;       /* staged K1: sum of the sorted-segment kernels' durations (clean with serial passes) */
    float sort_ms;         /* staged K1: sum of the key sorts' durations (clean with serial passes)             */
    uint32_t sorted_stages; /* staged K1: sorted stages per pass of the render                                  */
    uint32_t queue_entries; /* staged K1: entries each queue buffer holds (= paths per pass)                    */
} RzTiming;

typedef struct RzContext RzContext;

uint32_t rayz_cuda_abi_version(void);

/* Lifetime.  Replaces Tracer.init's allocation of img/hittables/bvh (renderer.zig:29-64). */
int rayz_cuda_create(const RzConfig *cfg, RzContext **out);
void rayz_cuda_destroy(RzContext *ctx);

/* Launch on a caller-owned CUDA stream (a cudaStream_t passed as void*) of device 0 of the
 * context instead of the library's own; NULL restores the library stream. */
int rayz_cuda_set_stream(RzContext *ctx, void *cuda_stream);

/* Replaces pool.initHittables + bvh.build (renderer.zig:76-78, ecs.zig:43-51, hit.zig:130-161):
 * flattens the scene to device SoA buffers on every device and builds the device BVHs. */
int rayz_cuda_upload_scene(RzContext *ctx, const RzScene *scene);

/*
 * THE HOT PATH.  Replaces the pixel loop of Tracer.render (renderer.zig:80-97) and the
 * sqrt/clamp/u8 of writePPM (image.zig:35-38).  Blocking.  Host outputs (each nullable):
 *   out_linear_rgba : rows_of_shard * width * 4 floats, linear radiance mean (a = 1)
 *   out_rgb8        : rows_of_shard * width * 3 bytes, trunc(255*clamp(sqrt(x),0,1))
 *   out_paths       : rows_of_shard * width * spp  (the `usize` render() returns, :100)
 */
int rayz_cuda_render(RzContext *ctx, const RzCamera *cam, const RzRenderParams *params,
                     float *out_linear_rgba, uint8_t *out_rgb8, uint64_t *out_paths);

/* Optional: allocate everything a render with these parameters needs (accumulators, result buffers, the
 * staged K1's queues: up to ~31 GB at the default pass size) ahead of time, like Image.initEmpty in Tracer.init (renderer.zig:29-64),
 * so that the first rayz_cuda_render does not pay for it. */
int rayz_cuda_reserve(RzContext *ctx, const RzRenderParams *params);

/* Same, but results stay in HBM on device_ids[0]; pointers (valid until the next render or
 * destroy) are returned instead of copied.  With `sync` == 0 the call only enqueues. */
int rayz_cuda_render_device(RzContext *ctx, const RzCamera *cam, const RzRenderParams *params,
                            void **d_linear_rgba, void **d_rgb8, uint64_t *out_paths, int sync);

/*
 * Per-pixel noise of the accumulated frame of the last render(s): the standard error of the displayed value
 *   Ybar = (0.2126 q0 + 0.7152 q1 + 0.0722 q2) / n,  s^2 = (q3 / n - Ybar^2) n / (n - 1)  (q: per-pixel sums, n: samples),
 *   e = sqrt(s^2 / n) / (2 sqrt(max(Ybar, 1e-4)))
 * out_err (nullable): rows of the context * width floats, laid out like out_linear_rgba.  out (nullable): the frame summary,
 * n_above counting pixels with e > target.  RZ_ERR_INVALID_ARG unless the accumulated render(s) ran with RZ_RENDER_MOMENTS.
 */
int rayz_cuda_noise(RzContext *ctx, float target, float *out_err, RzNoise *out);

/*
 * Render until the frame is clean enough: the first batch is p->spp samples from p->sample_offset (RZ_RENDER_MOMENTS
 * implied), each next batch doubles the accumulated count (capped at max_spp) with RZ_RENDER_ACCUMULATE; stops when
 * rms_err <= target or max_spp samples are reached.  RZ_OK either way: *out_noise says which (its samples and rms_err).
 * The host buffers (each nullable, as in rayz_cuda_render) are written once, at the end; *out_paths counts every batch.
 * RZ_ERR_INVALID_ARG if max_spp < p->spp.
 */
int rayz_cuda_render_to_noise(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, float target, uint32_t max_spp,
                              float *out_linear_rgba, uint8_t *out_rgb8, uint64_t *out_paths, RzNoise *out_noise);

/* Number of image rows a shard owns under the banding rule above. */
uint32_t rayz_cuda_shard_rows(uint32_t height, uint32_t shard_index, uint32_t shard_count,
                              uint32_t band_rows);

/* Rows a CONTEXT renders (= rows of the out_* buffers of rayz_cuda_render) when it is shard
 * `shard_index` of `shard_count`: a context with n devices deals its share to them as shards
 * shard_index*n .. shard_index*n + n-1 of shard_count*n.  Equals rayz_cuda_shard_rows for n = 1. */
uint32_t rayz_cuda_context_rows(const RzContext *ctx, uint32_t height, uint32_t shard_index,
                                uint32_t shard_count, uint32_t band_rows);

/* K0: f64, FMA-free closest-hit sphere index of the deterministic pixel-centre ray
 * getRay(i, j, null) (camera.zig:59-77) through the reference's BVH order
 * (hit.zig:181-216).  out_ids: width*height int32, -1 = miss.  use_bvh = 0 => brute force. */
int rayz_cuda_primary_ids(RzContext *ctx, const RzCamera *cam, uint32_t width, uint32_t height,
                          int use_bvh, int32_t *out_ids);

int rayz_cuda_stats(RzContext *ctx, RzStats *out);

/* The same counters per stage of the staged K1 (RZ_VARIANT_MEGA): 0 = primary kernel (camera segments),
 * 1 = sorted stages, 2 = persistent tail kernel.  Other variants count everything under stage 0. */
int rayz_cuda_stage_stats(RzContext *ctx, uint32_t stage, RzStats *out);
int rayz_cuda_timing(RzContext *ctx, RzTiming *out);

/* K6: dependent-free FFMA chains on every SM of device 0; returns achieved FP32 TFLOP/s
 * (2 flop per FFMA) over ~`millis` ms and the SM count. Roofline denominator. */
int rayz_cuda_fp32_peak(RzContext *ctx, uint32_t millis, double *out_tflops, int32_t *out_sms);

/*
 * Tuning (experiments and tests; every field has a measured default, DESIGN.md sections 3 and 5).  Not part of the
 * reference-facing contract: the reference has no such knobs.  Read the current values, change what you want, set.
 * The library reads NO environment variables.
 */
typedef struct RzTuning {
    uint32_t struct_size;     /* sizeof(RzTuning) of the caller (checked)                                              */
    int32_t rays_per_thread;  /* K1b / wavefront: independent paths per lane, 1 or 2 (default 2)                        */
    uint32_t chunk;           /* samples per work unit (32 pixels x chunk) of the persistent kernels (default 16)       */
    uint32_t chunk_primary;   /* ... of the camera-stage kernels (K1a, staged K3), which build a culled list per unit (64) */
    int32_t queue_log2;       /* staged K1: queue entries per pass = 2^queue_log2, 16..28 (default 27: 6.4 GB per queue
                               * buffer; 28 is ~2 % faster on 405 M-path renders and doubles the reservation)           */
    int32_t second_stages;    /* staged K1: sorted stages after the camera segment, 0..8; -1 = automatic (default)      */
    int32_t bvh_stages;       /* staged BVH kernel: sorted stages, 0..8 (default 0: measured as a loss)                 */
    int32_t tail_brute;       /* staged K1: 1 = the tail of the paths stays brute force (default 0: BVH kernel)         */
    int32_t bvh_staged;       /* BVH variant: 1 = FRAMES of >= 2^26 paths run a camera stage + queue first (default 1)  */
    int32_t cell_bits;        /* sort key: bits of the origin cell, 0..9 (default 9)                                    */
    int32_t bvh_active_min;   /* K3: lanes that must still traverse for a burst to go on, 1..32 (default 8)             */
    int32_t bvh_descend_min;  /* K3: a descend round ends below this many descending lanes (default 24)                 */
    int32_t sah_leaf;         /* host SAH builder: max spheres per leaf, 1..8 (default 4); applies at the next upload   */
    double sah_node_cost;     /* host SAH builder: cost of a node visit relative to a sphere test (default 0.5)         */
    uint32_t unit_entries;    /* sorted-stage kernel: queue entries per work unit (upper bound; small stages use
                               * fewer), 64..2048, multiple of 64 (default 512: 4 bytes of shared memory per entry and
                               * warp; 1024 costs a resident CTA)                                                       */
    uint32_t debug_queue_cap; /* tests: pretend the queues hold only this many entries (0 = off) -> RZ_ERR_INTERNAL     */
    uint32_t debug_stack_cap; /* tests: pretend the K3 traversal stack holds only this many entries (0 = off)           */
    int32_t key_sectors;      /* sort key direction field: 0 = octant, 1 = 45-degree sector in the plane of the sphere
                               * box's two long axes, 2 = 22.5-degree sector (and one cell bit less), -1 = 45-degree
                               * sectors when that box is flat, octants otherwise (default)                              */
    int32_t lbvh_leaf;        /* device LBVH builder: subtrees of at most this many spheres become one leaf, 1..8
                               * (default 1: 4 makes 6.5 sphere tests per segment instead of 1.5 for 6 fewer box tests); applies at the next upload                                */
    double huge_factor;       /* staged K1: spheres above huge_factor x the median radius (at most max(4, n/32) of them)
                               * stay outside the box the sort key's cells and reach classes are measured in, and are
                               * culled by direction only (default 4: the r = 1000 ground and the three r = 1 spheres of
                               * the reference scenes; 8 keeps the latter inside: +40-60 % sphere tests per sorted
                               * segment); applies at the next upload                                                    */
} RzTuning;
int rayz_cuda_get_tuning(RzContext *ctx, RzTuning *out);
int rayz_cuda_set_tuning(RzContext *ctx, const RzTuning *tuning);

const char *rayz_cuda_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* RAYZ_CUDA_H */
