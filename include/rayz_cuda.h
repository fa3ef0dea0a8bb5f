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
                                    * seed, max_depth, t_min, camera, RZ_RENDER_MOMENTS, RZ_RENDER_SOBOL, RZ_RENDER_RQMC and RZ_RENDER_PASSES bits on this context, no scene
                                    * upload or differently shaped reserve (or an RZ_RENDER_RQMC reserve after a render without
                                    * the flag, which grows the accumulators) came in between, sample_offset equals the previous
                                    * batch's sample_offset + spp, and the cumulative count stays below 2^32.  A render that
                                    * fails ends the accumulation.  *out_paths counts this call's paths only.  With
                                    * rayz_cuda_render_device(sync = 0), the next batch checks the previous one's device
                                    * error word before it adds to its sums. */
#define RZ_RENDER_ADAPTIVE 0x8u    /* adaptive sampling, honoured by rayz_cuda_render_to_noise only (rayz_cuda_render and
                                    * rayz_cuda_render_device refuse it with RZ_ERR_INVALID_ARG; rayz_cuda_reserve also allocates
                                    * the per-pixel counts and lists, 8 bytes per pixel).  The doubling schedule runs per pixel:
                                    * after the first round, a round traces only the pixels that took part in every earlier round
                                    * and whose error (as rayz_cuda_noise's out_err shows it) is above the target.  A pixel that
                                    * ends with c samples equals the same pixel of a uniform c-spp render bit for bit (linear,
                                    * rgb8, error), as every path is a function of (seed, pixel, sample index).  AUTO runs the BVH
                                    * family; a pinned MEGA, MEGA_SINGLE or WAVEFRONT runs its first round as pinned and the
                                    * others with the single-form brute-force kernel (the same family: for exactness, not speed).
                                    * Whether a pixel is active depends on its own sums only (under RZ_RENDER_RQMC, on them and on
                                    * its row segment's gain, which no shard splits), so sharding changes no count.
                                    * rayz_cuda_noise and rayz_cuda_pixel_samples read the frame with each pixel's own count; an
                                    * RZ_RENDER_ACCUMULATE batch after it is refused, the sums untouched. */
#define RZ_RENDER_SOBOL 0x10u      /* low-discrepancy sampling (DESIGN.md "Low-discrepancy sampling"): the camera's and each
                                    * scatter's uniforms come from 2-D pairs of an Owen-scrambled Sobol sequence instead of
                                    * independent Philox draws.  Pairs: camera A = jitter (x, y); camera B = lens (radius, angle,
                                    * area-preserving polar map); camera C = shutter time (first coordinate); bounce s = 1..max_depth
                                    * = the scatter's u.x, u.y (the sphere direction; u.x is also the dielectric's Fresnel choice).
                                    * u.z and u.w of a bounce stay Philox.  Construction (Burley 2020, "Practical Hash-based Owen
                                    * Scrambling", with padding): point i of a pair is (Sobol dimension 0, dimension 1) of the
                                    * shuffled index i' = S(i, s_shuffle), each coordinate then scrambled x = S(x, s_dim), with S a
                                    * nested-uniform (Owen) scramble (bit reversal, Laine-Karras-style hash keyed by s, bit
                                    * reversal); dimension 0 = the bit-reversed index, dimension 1 = Joe-Kuo d = 2 (s = 1, a = 0,
                                    * m = {1}); the top 24 bits become the uniform.  The seeds s are an integer hash of (seed, global
                                    * pixel, pair) only, so every uniform is still a pure function of (seed, global pixel, sample
                                    * index, bounce) and every guarantee above holds as written: sharding, batches, adaptive pixels,
                                    * guides.  Stratification: for each pixel and pair, the 2^k points of an aligned sample block
                                    * [m 2^k, (m + 1) 2^k) form a (0,k,2)-net: for every a + b = k each box of 2^-a x 2^-b holds
                                    * exactly one point (the doubling schedule of rayz_cuda_render_to_noise hands out such blocks from
                                    * a power-of-two start).  The noise estimate (rayz_cuda_noise) keeps its formula, which assumes
                                    * independent samples: with this flag the error of the mean is expected to be smaller than it
                                    * says (conservative), so rayz_cuda_render_to_noise stops about where it would without the flag;
                                    * the gain shows in fixed-spp frames and in the denoiser's input.  RZ_RENDER_RQMC makes the
                                    * estimate see the gain. */
#define RZ_RENDER_RQMC 0x20u       /* randomised-QMC noise estimate over RZ_RENDER_SOBOL (DESIGN.md "Low-discrepancy sampling",
                                    * "The RQMC estimate").  Requires RZ_RENDER_SOBOL and RZ_RENDER_MOMENTS (rayz_cuda_render_to_noise
                                    * implies MOMENTS, so there it needs SOBOL only), an even spp and sample_offset, and in
                                    * rayz_cuda_render_to_noise an even max_spp; anything else is refused with RZ_ERR_INVALID_ARG,
                                    * the message naming the rule, nothing touched.  An RZ_RENDER_ACCUMULATE batch whose RQMC bit
                                    * differs from the accumulated render's is refused, the sums untouched.
                                    * Replicates (R = 2): sample index i belongs to replicate r = i & 1 and is that replicate's sample
                                    * j = i >> 1.  Each replicate is an Owen-scrambled Sobol sequence as above with its own seeds: the
                                    * pair's base seed b = rz_sobol_pair_seed(seed, global pixel, pair) becomes
                                    * b_r = rz_hash32(b ^ (0x9e3779b9 + r)), and point i is point j of the pair under b_r.  Every
                                    * uniform is still a pure function of (seed, global pixel, sample index, bounce): sharding,
                                    * batches, adaptive pixels and guides keep their guarantees.  Within each replicate the aligned
                                    * blocks of j are (0,k,2)-nets.  The image and rayz_cuda_pixel_samples do not change meaning:
                                    * a pixel is the mean of all n samples.
                                    * The estimate.  A sky path adds its clamped luminance Y (rz_luma_sq's Y) in 2^-32 fixed point to
                                    * its replicate's sum Q_r (16 bytes a pixel).  For a pixel with n samples, m = n / 2:
                                    *   mu_r = Q_r 2^-32 / m,  V_rep = (mu_0 - mu_1)^2 / 4  (sum_r (mu_r - mu)^2 / (R (R - 1)), R = 2),
                                    *   V_iid = s^2 / n  (the s^2 of the error formula of RzNoise / rayz_cuda_noise).
                                    * A segment is the pixels of one global row with x in [64k, 64k + 64) (the last one of a row may be
                                    * shorter); G = sum_seg V_rep / sum_seg V_iid, 1 when the denominator is 0, not clamped; and the
                                    * pixel's error is e = e_iid sqrt(G), with the G of its segment when the pixel's count was last
                                    * the frame's largest: in a uniform frame, the current G of every pixel; under RZ_RENDER_ADAPTIVE,
                                    * the G its last stopping test read, so that a pixel that stopped keeps the error it stopped at
                                    * while its segment's other pixels take more samples, and max_err <= target unless capped holds
                                    * as without the flag.  One pixel's V_rep has one degree of freedom; a segment pools
                                    * about 64, so sqrt(G) is good to about +-9 %, while the per-pixel shape comes from the iid term.
                                    * Segments lie inside a global row, which no shard or device splits: e and every adaptive count
                                    * are shard- and device-invariant.  This e is what out_err, the summary and n_above of
                                    * rayz_cuda_noise, both tests of rayz_cuda_render_to_noise and the denoiser's v_p use.
                                    * Trade-off: two replicates of n / 2 points carry more variance than one sequence of n points, so
                                    * the frame itself is somewhat noisier than under RZ_RENDER_SOBOL alone; hence a separate flag. */
#define RZ_RENDER_ADAPTIVE_POOLED 0x40u /* pooled adaptive stopping (DESIGN.md "Adaptive sampling", "Pooled stopping"): honoured
                                    * by rayz_cuda_render_to_noise together with RZ_RENDER_ADAPTIVE only; without ADAPTIVE, and in
                                    * rayz_cuda_render, rayz_cuda_render_device and rayz_cuda_render_guides, it is refused with
                                    * RZ_ERR_INVALID_ARG, the message naming the rule, nothing touched (rayz_cuda_reserve takes it
                                    * with ADAPTIVE).  The plain rule stops a pixel on its own iid estimate, which after 4 or 16
                                    * samples is itself very noisy: the pixels that stop early are those whose estimate came out
                                    * low, and the measured error of the frame is several times the target.  Under this flag a
                                    * pixel's per-sample variance is shrunk toward its row segment's (the segment of RZ_RENDER_RQMC:
                                    * the pixels of one global row with x in [64k, 64k + 64), the last one of a row may be shorter).
                                    * For a pixel with n samples, e its rz_pixel_err (the formula of rayz_cuda_noise), u = n e^2,
                                    * d = n - 1:
                                    *   U_S = sum d_i u_i / sum d_i over the segment's pixels with n_i >= 2 (0 if there are none),
                                    *   e* = sqrt((NU0 U_S + d u) / (NU0 + d) / n)   (+inf while n < 2),  NU0 = 16,
                                    * and under RZ_RENDER_RQMC e* sqrt(G).  NU0 is the prior's weight in degrees of freedom, chosen
                                    * by measurement (DESIGN.md).  U_S is frozen like G: a pixel keeps the U_S its last stopping
                                    * test read, so that a pixel that stopped keeps the error it stopped at while its segment's
                                    * other pixels take more samples.  e* is what out_err, the summary and n_above of
                                    * rayz_cuda_noise, the stopping test and the denoiser's v_p use, so max_err <= target unless
                                    * samples == max_spp holds as written; rayz_cuda_noise, rayz_cuda_pixel_samples and
                                    * rayz_cuda_denoise after the call read e*.  A pixel's activity now depends on its segment's
                                    * sums as well as its own (a lucky pixel in a noisy segment cannot stop on a few agreeing
                                    * samples; a pixel of a clean segment still stops early); segments lie inside a global row,
                                    * which no shard or device splits, so every count, the image and e* stay shard- and
                                    * device-invariant.  Costs: 8 bytes per pixel and one double per segment, and one warp per
                                    * segment before each stopping test (the pass RZ_RENDER_RQMC's gain runs in); the path kernels
                                    * are those of the plain rule, and more samples are spent where the plain rule stopped too
                                    * early. */
#define RZ_RENDER_PASSES 0x80u     /* light-path passes (DESIGN.md "Light-path passes"): also sum each path's radiance into the
                                    * one pass (RZ_PASS_*, below) its path belongs to, so that rayz_cuda_passes can split every
                                    * pixel by how its light reached the sky.  Changes no pixel of the image and no noise estimate.
                                    * Honoured by rayz_cuda_render, rayz_cuda_render_device and rayz_cuda_render_to_noise (plain,
                                    * adaptive and pooled), by every variant and sampler; rayz_cuda_reserve also allocates the pass
                                    * sums (RZ_PASS_COUNT x 3 x 8 = 168 bytes per pixel).  An RZ_RENDER_ACCUMULATE batch whose
                                    * PASSES bit differs from the accumulated render's is refused, the sums untouched;
                                    * rayz_cuda_render_guides refuses the flag; max_depth > 2^29 - 1 is refused with
                                    * RZ_ERR_INVALID_ARG (the first hit's kind rides in the top bits of a path's hit count). */
/* Pixel reconstruction filter (DESIGN.md "Pixel filters"), a field of flags: the kind in bits 8-9, the width in bits 16-23.
 * Filter importance sampling: each camera sample's offset from the pixel centre is drawn from the filter, and the sample keeps
 * weight 1.  Sample (px, py) with jitter uniforms (ux, uy) (Philox, or Sobol's camera-jitter pair) starts at
 * (px + w(ux), py + w(uy)), w the inverse CDF of the filter's normalised marginal g; lens, time and scatter uniforms are
 * unchanged.  The filters are separable, f(x, y) = g(x) g(y), with support |x| <= R = W / 2 for the full width W:
 *   RZ_FILTER_BOX              w(u) = u - 0.5 (the reference's getRay jitter, bit for bit the code path without the field)
 *   RZ_FILTER_TENT             g(x) = 1 - |x| / R                                                       default W = 2 px
 *   RZ_FILTER_GAUSSIAN         g(x) = exp(-x^2 / 2 s^2) - exp(-R^2 / 2 s^2), s = W / 6 (pbrt-v4's form)  default W = 3 px
 *   RZ_FILTER_BLACKMAN_HARRIS  g(x) = 0.35875 + 0.48829 cos(2 pi x / W) + 0.14128 cos(4 pi x / W)
 *                                     + 0.01168 cos(6 pi x / W) (Cycles' form)                          default W = 1.5 px
 * The width field is W in 1/16 px: 0 is the kind's default, otherwise 16..64 (1 to 4 px).  w is monotone in u, inside [-R, R]
 * and odd about u = 1/2, and within 1e-5 px of the exact inverse CDF at every 24-bit u (interpolated in f64 from exact tables
 * of the unit-width filter, rounded to f32 once).
 * Every sample keeps weight 1 and a pixel stays the mean of its own samples: batches, shards, devices, adaptive counts, passes
 * and the noise estimate keep every guarantee they have with the box.  Under RZ_RENDER_SOBOL the warp is monotone per axis, so
 * each stratum of the jitter pair maps to a box of equal filter mass.  Honoured by rayz_cuda_render, rayz_cuda_render_device,
 * rayz_cuda_render_to_noise (plain, adaptive and pooled), rayz_cuda_render_guides and rayz_cuda_render_mattes, with every
 * variant and sampler; rayz_cuda_primary_ids (pixel centres) ignores it.  Refused with RZ_ERR_INVALID_ARG, the message naming
 * the rule and nothing touched: a width of 1..15 or above 64, a nonzero width with RZ_FILTER_BOX, and an RZ_RENDER_ACCUMULATE
 * batch whose field (kind or width) differs from the accumulated render's.  rayz_cuda_denoise refuses guide buffers rendered
 * with another field than the accumulated frame. */
#define RZ_RENDER_FILTER_SHIFT 8
#define RZ_RENDER_FILTER_MASK 0x300u
#define RZ_RENDER_FILTER_WIDTH_SHIFT 16
#define RZ_RENDER_FILTER_WIDTH_MASK 0xff0000u
#define RZ_FILTER_BOX 0u
#define RZ_FILTER_TENT 1u
#define RZ_FILTER_GAUSSIAN 2u
#define RZ_FILTER_BLACKMAN_HARRIS 3u
#define RZ_FILTER_WIDTH_MIN 16u   /* 1 px, in 1/16 px */
#define RZ_FILTER_WIDTH_MAX 64u   /* 4 px */
/* the flags of a filter: kind RZ_FILTER_*, width16 the full width in 1/16 px (0: the kind's default) */
#define RZ_RENDER_FILTER(kind, width16) \
    ((((uint32_t)(kind) << RZ_RENDER_FILTER_SHIFT) & RZ_RENDER_FILTER_MASK) | \
     (((uint32_t)(width16) << RZ_RENDER_FILTER_WIDTH_SHIFT) & RZ_RENDER_FILTER_WIDTH_MASK))

/*
 * Light-path passes (RZ_RENDER_PASSES).  A path that ends in the sky with h scattering hits before it adds its clamped
 * radiance, the same 2^-32 fixed-point values the three colour accumulators add, to exactly one pass:
 *   RZ_PASS_ENVIRONMENT                                  h = 0 (the camera ray missed)
 *   RZ_PASS_DIFFUSE_DIRECT / RZ_PASS_DIFFUSE_INDIRECT    first hit RZ_MAT_DIFFUSE;    h = 1 / h >= 2
 *   RZ_PASS_GLOSSY_DIRECT / RZ_PASS_GLOSSY_INDIRECT      first hit RZ_MAT_METALLIC;   h = 1 / h >= 2
 *   RZ_PASS_TRANSMISSION_DIRECT / _INDIRECT              first hit RZ_MAT_DIELECTRIC (whether it reflected or refracted);
 *                                                        h = 1 / h >= 2
 * The class is decided by the first hit's MATERIAL KIND, not by the lobe its scatter took: a dielectric hit that reflects
 * still counts as transmission.  Paths that end absorbed or at the depth limit add nothing to any pass, as they add nothing
 * to the image.  Since every path adds the same integers to its pass as to the image, for every pixel and channel the sum of
 * the seven pass sums equals the image's sum bit for bit, through batches, shards, devices and adaptive rounds.
 */
enum {
    RZ_PASS_ENVIRONMENT = 0,
    RZ_PASS_DIFFUSE_DIRECT = 1,
    RZ_PASS_DIFFUSE_INDIRECT = 2,
    RZ_PASS_GLOSSY_DIRECT = 3,
    RZ_PASS_GLOSSY_INDIRECT = 4,
    RZ_PASS_TRANSMISSION_DIRECT = 5,
    RZ_PASS_TRANSMISSION_INDIRECT = 6,
    RZ_PASS_COUNT = 7
};

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
 * With RZ_RENDER_ADAPTIVE in p->flags, `target` bounds EACH pixel's error instead of the rms: with N the count after a
 * round, the next round gives the pixels still active (count N, error > target) the samples [N, N + b) past sample_offset,
 * b = min(N, max_spp - N); the call ends when no pixel is active or N reaches max_spp.  *out_paths is the sum of the per-pixel
 * counts; *out_noise is over all pixels, each with its own count, and its samples is the largest count: max_err <= target
 * unless samples == max_spp.  RzStats and RzTiming describe the last round, except total_ms, which covers the call.
 */
int rayz_cuda_render_to_noise(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, float target, uint32_t max_spp,
                              float *out_linear_rgba, uint8_t *out_rgb8, uint64_t *out_paths, RzNoise *out_noise);

/*
 * Per-pixel sample counts of the accumulated frame: out_spp holds rows of the context * width counts, laid out like
 * rayz_cuda_noise's out_err.  After a uniform render (or batches) every count is the frame's; after an adaptive
 * rayz_cuda_render_to_noise, each pixel's own.  RZ_ERR_INVALID_ARG if there is no accumulated render.
 */
int rayz_cuda_pixel_samples(RzContext *ctx, uint32_t *out_spp);

/*
 * Light-path passes of the accumulated frame (RZ_RENDER_PASSES).  out_passes holds RZ_PASS_COUNT planes of rows of the context
 * * width * 4 floats, plane i at out_passes + i * rows * width * 4, each laid out like out_linear_rgba: rgb = the pass sum over
 * the pixel's own sample count (n_px after an adaptive rayz_cuda_render_to_noise), in the resolve's f64 arithmetic, stored as
 * f32; a = 1.  Their sum equals out_linear_rgba to f32 rounding.  RZ_ERR_INVALID_ARG, nothing touched, if out_passes is NULL,
 * there is no accumulated frame or it was rendered without RZ_RENDER_PASSES.  Leaves the accumulated frame, its sample counts,
 * RzStats, RzTiming and rayz_cuda_render_device's buffers untouched (a render enqueued by rayz_cuda_render_device(sync = 0) is
 * waited for first, as rayz_cuda_noise does).
 */
int rayz_cuda_passes(RzContext *ctx, float *out_passes);

/*
 * Guide buffers for a denoiser, of the camera samples [p->sample_offset, p->sample_offset + p->spp) of every pixel of the
 * context's rows: the SAME camera rays (seed, global pixel, sample index -> jitter, lens point, time) a render with these
 * parameters traces, each followed to its first hit only.  Host outputs, each nullable, laid out like out_linear_rgba:
 *   out_albedo : rows * width * 4 floats: rgb = mean over all samples of the first hit's albedo,
 *                a = coverage (fraction of samples that hit a sphere)
 *   out_normal : rows * width * 4 floats: xyz = mean over all samples of the hit's unit normal (facing the ray, 0 for a miss),
 *                w = mean hit distance over the samples that hit (0 if none did)
 * Per sample: albedo = the texture colour at the f64-refined hit point for diffuse and metallic materials (the attenuation of
 * their scatter, also where a metal's scatter would be absorbed), (1, 1, 1) for dielectrics, the sky colour of the ray's
 * direction for a miss; normal = the unit normal of the hit in world space, flipped against the ray; distance = the hit's t
 * along the unit camera ray from its lens-sampled origin.  Each pixel's samples are summed in f64 in sample order and the f32
 * mean is written, so the buffers depend on (scene, camera, seed, pixel, sample range) only: not on shards, devices or launch
 * shape.  The search is the BVH kernel's (RZ_VARIANT_BVH) whatever the variant; max_depth and collect_stats have no effect.
 * Parameters a render refuses are refused with its codes and messages, prefixed "guides:"; RZ_RENDER_ACCUMULATE,
 * RZ_RENDER_ADAPTIVE and RZ_RENDER_PASSES are refused with RZ_ERR_INVALID_ARG.  RZ_ERR_INTERNAL if the traversal stack overflowed (results withheld,
 * the context stays usable).  Leaves the accumulated frame, its sample counts, RzStats and RzTiming untouched (a render
 * enqueued by rayz_cuda_render_device(sync = 0) is waited for first, as rayz_cuda_noise does).
 */
int rayz_cuda_render_guides(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, float *out_albedo, float *out_normal);

/*
 * ID mattes, for compositing (the data Cryptomatte stores): per pixel of the context's rows, the spheres its camera samples
 * [p->sample_offset, p->sample_offset + p->spp) hit first, ranked by exact coverage.  The samples are the SAME camera rays a
 * render with these parameters traces and rayz_cuda_render_guides follows (jitter, lens point, shutter time, every sampler),
 * each followed to its first hit by the BVH kernel's search.  A sample's id is the caller's index of that sphere
 * (RzScene order), or RZ_MATTE_MISS for a miss.  n_id = the pixel's samples with that id.  Ranks are ordered by n_id
 * descending, then id ascending: a total order, so the result depends on (scene, camera, seed, pixel, sample range) only, not
 * on shards, devices or launch shape.  Host outputs, each nullable, of rows * width * ranks entries, rank r of local pixel lp at
 * lp * ranks + r (rows ordered like out_linear_rgba):
 *   out_ids      : the id of the rank, RZ_MATTE_EMPTY past the pixel's distinct ids
 *   out_coverage : (float)((double)n_id / (double)spp), 0 past the pixel's distinct ids
 * Counts are recoverable exactly as rint(coverage * spp); with ranks >= spp the ranks hold the pixel's whole histogram.
 * max_depth and collect_stats have no effect.  Refused with nothing touched, messages prefixed "mattes:": RZ_ERR_INVALID_ARG for
 * NULL ctx, cam or p, ranks of 0 or above RZ_MATTE_MAX_RANKS, spp above RZ_MATTE_MAX_SPP, and RZ_RENDER_ACCUMULATE,
 * RZ_RENDER_ADAPTIVE, RZ_RENDER_ADAPTIVE_POOLED or RZ_RENDER_PASSES in the flags; parameters a render refuses, with its codes.
 * RZ_ERR_INTERNAL if the traversal stack overflowed (results withheld, the context stays usable).  Leaves the accumulated frame,
 * its sample counts, the guide buffers, RzStats, RzTiming and rayz_cuda_render_device's buffers untouched (a render enqueued by
 * rayz_cuda_render_device(sync = 0) is waited for first, as rayz_cuda_render_guides does).
 */
#define RZ_MATTE_MISS   (-1)    /* id of a camera sample that hit no sphere (the sky)              */
#define RZ_MATTE_EMPTY  (-2)    /* id of a rank past the pixel's distinct ids; its coverage is 0   */
#define RZ_MATTE_MAX_RANKS 16u
#define RZ_MATTE_MAX_SPP 1024u
int rayz_cuda_render_mattes(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, uint32_t ranks,
                            int32_t *out_ids, float *out_coverage);

/*
 * Denoiser parameters (rayz_cuda_denoise).  A zero sigma takes its default.
 */
typedef struct RzDenoiseParams {
    uint32_t struct_size;  /* sizeof(RzDenoiseParams) of the caller (checked, like RzTuning)                       */
    uint32_t iterations;   /* à-trous levels, step 2^k for k = 0..iterations-1; 0..10; 0 = the input unchanged     */
    float sigma_luminance; /* 0 => 4    */
    float sigma_normal;    /* 0 => 128  */
    float sigma_depth;     /* 0 => 1    */
    uint32_t reserved0;
} RzDenoiseParams;

/*
 * Denoised accumulated frame of the last render(s): an edge-avoiding à-trous filter (SVGF's spatial filter, Schied et al. 2017;
 * Dammertz et al. 2010) steered by the per-pixel noise estimate and the guide buffers of the last successful
 * rayz_cuda_render_guides call.  dp == NULL: 5 iterations and the default sigmas.  Host outputs, each nullable, laid out like
 * rayz_cuda_render's: out_linear_rgba (a = 1) and out_rgb8 = trunc(255 clamp(sqrt(x), 0, 1)) of that f32 linear value in f64.
 * Per pixel p, with Y(x) = 0.2126 x.r + 0.7152 x.g + 0.0722 x.b, c_p the resolved linear rgb (each pixel's own count after an
 * adaptive render), e_p rayz_cuda_noise's error and a_p, n_p, z_p the guide albedo, normal and depth:
 *   v_p = 4 e_p^2 max(Y(c_p), 1e-4)                         (variance of the pixel mean's luminance; e = +inf gives +inf)
 *   i_p = c_p / max(a_p, 1e-3) per channel,  v_p /= max(Y(a_p), 1e-3)^2                             (demodulation)
 *   g_p = ((z[x+1] - z[x-1]) / 2, (z[y+1] - z[y-1]) / 2), indices clamped at the frame edges (once per call)
 *   level k, step s = 2^k, taps q = p + s (dx, dy), dx, dy in -2..2 (taps outside the frame skipped), h = (1, 4, 6, 4, 1) / 16:
 *     gv_p = the 3 x 3 (1, 2, 1) binomial blur of the current v around p (taps outside the frame skipped, renormalised)
 *     w_l  = exp(-|Y(i_p) - Y(i_q)| / (sigma_luminance sqrt(gv_p) + 1e-4))                     (1 when gv_p = +inf)
 *     w_n  = clamp(n_p.n_q / (|n_p| |n_q|), 0, 1)^sigma_normal if both normals are nonzero, 1 if both are zero (sky), else 0
 *     w_z  = exp(-|z_p - z_q| / (sigma_depth |g_p . (q - p)| + 1e-2))
 *     w    = h[dx] h[dy] w_l w_n w_z,   i'_p = sum w i_q / sum w,   v'_p = sum w^2 v_q / (sum w)^2 (a tap whose f32 w^2 is 0
 *            adds nothing to the variance)
 *   out_p = i_p max(a_p, 1e-3)                                                                        (remodulation)
 * iterations = 0 returns the resolved frame exactly (rayz_cuda_render's linear and rgb8 of the accumulated frame).  The filter
 * runs in f32 on the gather root (device_ids[0]) over the whole frame, so every device count gives the same bytes.  The guides'
 * sample range need not match the render's (cheap 16-spp guides under a 500-spp render are the intended use).
 * Refused, nothing touched, with messages prefixed "denoise:": RZ_ERR_INVALID_ARG for a bad struct_size, iterations > 10 or a
 * negative or non-finite sigma, no accumulated frame, one rendered without RZ_RENDER_MOMENTS, no guide buffers (none, the last
 * guides call failed, or a scene upload or a reserve of another frame came in between) or guides whose frame, camera or seed
 * differ from the accumulated frame's; RZ_ERR_UNSUPPORTED for a shard (shard_count > 1: its rows are not image neighbours).
 * Leaves the accumulated frame, its sample counts, RzStats, RzTiming and rayz_cuda_render_device's buffers untouched (a render
 * enqueued by rayz_cuda_render_device(sync = 0) is waited for first, as rayz_cuda_noise does).
 */
int rayz_cuda_denoise(RzContext *ctx, const RzDenoiseParams *dp, float *out_linear_rgba, uint8_t *out_rgb8);

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
