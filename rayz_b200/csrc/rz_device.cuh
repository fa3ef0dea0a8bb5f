// rz_device.cuh — device-side types, counter-based RNG and the shading half of the path kernel.
//
// Everything here is `RZ_HD` (host+device) so that tests/hostsim can compile the very same
// FP32 shading code for the CPU and compare its statistics with the f64 oracle in a container
// that has no GPU.  That host build is test infrastructure; the product only ever launches the
// CUDA kernels (rz_path.cu etc.) and has no CPU path.
//
// Reference functions restated here (paths under /root/reference/src):
//   Camera.getRay + randomInDefocus   camera.zig:59-90     -> rz_camera_ray
//   Hit.init                          hit.zig:25-41        -> rz_refine_hit (front face flip)
//   Sphere.hitInner (accepted root)   geom.zig:38-66       -> rz_refine_hit (f64 re-evaluation)
//   Texture.value / CheckerTexture    material.zig:19-51   -> rz_texture
//   Diffuse/Metallic/Dielectric       material.zig:73-160  -> rz_scatter
//   reflectance/reflect/refract       material.zig:179-194
//   bounceRay miss branch (sky)       renderer.zig:124-125 -> rz_sky
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <vector>

#define RZ_HD __host__ __device__ __forceinline__
// Rare branches of the shading code are kept OUT of line on the device: the staged kernels are 35-45 KB against a 32 KB L1.5
// instruction cache, and ncu charged up to 3 stall cycles per issued instruction to `no_instruction` (profiles/).
#ifdef __CUDA_ARCH__
#define RZ_COLD __device__ __noinline__
#else
#define RZ_COLD inline
#endif

// ---------------------------------------------------------------------------------------------
// Device scene: structure-of-arrays, one "sphere set" per kernel family (the brute-force set is
// ordered static-first, the BVH set in leaf order).  Index k below is the position in the set.
// ---------------------------------------------------------------------------------------------
struct RzSphereSet {
    const float4 *cr;      // [n_pad] (cx, cy, cz, -r^2)           FP32 intersection operand
    const float4 *vel;     // [n_pad] (vx, vy, vz, r)              Sphere.center.dir (geom.zig:12)
    const float4 *pk;      // brute set only: the same numbers pair-interleaved for the packed FP32x2
                           // search (rz_search_brute2): stationary pair p = spheres (2p, 2p+1) ->
                           // (cx0,cx1,cy0,cy1)(cz0,cz1,w0,w1), w = -r^2; moving pairs follow, each with
                           // two more float4 (vx0,vx1,vy0,vy1)(vz0,vz1,0,0).  n_static_pad + 2*n_moving_pad float4.
    const double4 *c64;    // [n]     (cx, cy, cz, r)  f64, for the refinement of the winning hit
    const double4 *v64;    // [n]     (vx, vy, vz, 1 / r)  f64
    const uint32_t *mat;   // [n]     material index (MaterialHandle.idx)
    const int32_t *orig;   // [n]     index in the caller's sphere array (ids, stats)
    uint32_t n;            // real spheres
    uint32_t n_static;     // spheres [0, n_static) are stationary            (brute set only)
    uint32_t n_static_pad; // static part padded to a multiple of 4           (brute set only)
    uint32_t n_pad;        // total padded count; moving part = [n_static_pad, n_pad)
};

struct RzMaterials {
    const uint32_t *kind;   // RZ_MAT_* (material.zig:162-165)
    const float *fuzz;      // min(fuzz, 1) is applied at scatter time (material.zig:112)
    const float *ior;
    const uint32_t *tex;
    const uint32_t *method; // RZ_DIFFUSE_* (material.zig:67-71)
    const float4 *rec;      // [4 * n_materials] the same facts flattened for the shading step, one 64-byte record per material:
                            //   (bits: kind | method << 2 | root-texture-is-solid << 4 | root-is-a-checker-of-two-solids << 5, fuzz, ior, bits: texture)
                            //   (r, g, b, 0 of a solid root, or of the checker's even texture) (r, g, b, 0 of its odd texture)
                            //   (1 / scale of the checker as the two halves of an f64, 0, 0)
                            // one load after set.mat[k] instead of a chain of dependent ones (kind -> tex -> tex kind -> 1/scale ->
                            // even / odd -> its kind -> colour: the checker ground of the reference scenes is half of all hits)
};

// What the shading step needs to know about a material (decoded RzMaterials::rec).
struct RzMatRec {
    uint32_t kind, method, tex;
    bool solid;      // the root texture is a solid colour: `color` is the attenuation, no texture walk
    bool checker2;   // the root texture is a checker of two solid colours: `color` (even) / `odd` by the lattice cell, no walk either
    float fuzz, ior;
    float3 color, odd;
    double inv_scale;
};

struct RzTextures {
    const uint32_t *kind;    // RZ_TEX_* (material.zig:41-43)
    const float4 *color;     // solid colour (rgb)
    const double *inv_scale; // 1 / CheckerTexture.scale
    const uint32_t *even;
    const uint32_t *odd;
};

// BVH2 node for the FP32 traversal kernel: both child boxes live in the parent so one 64-byte
// fetch decides both children.  As built: child < 0 => leaf: first = ~child, count in cnt.  As traversed (after
// rz_bvh_finalize): child = rz_leaf_ref(child, cnt) for leaves.
struct __align__(16) RzBvhNode {
    float lox[2], hix[2], loy[2], hiy[2], loz[2], hiz[2];
    int32_t child[2];
    uint32_t cnt[2];
};

// What the traversal kernel follows: an internal node's index (>= 0), or a leaf — ~((count - 1) << 28 | first), first < 2^28,
// count <= 8 — negative.  The builders write (child = ~first, cnt = count) for leaves; rz_bvh_finalize (rz_bvh_build.cu) turns
// every leaf's `child` into this reference once, at upload, and fills an unused slot (the root of a tiny scene) with a copy of
// its sibling, so that the node visit neither decodes nor checks anything.
RZ_HD int rz_leaf_ref(int child, uint32_t cnt) { return ~((int)((cnt - 1u) << 28) | ~child); }

struct RzCamF32 {
    float3 look_from, px_du, px_dv, px_origin, defocus_u, defocus_v;
    int defocus;
};

// bits of the device error word (RzPathArgs::err): a render that sets one returns RZ_ERR_INTERNAL
enum { RZ_DEV_ERR_QUEUE_OVERFLOW = 1u, RZ_DEV_ERR_STACK_OVERFLOW = 2u };

struct RzStatsDev {
    unsigned long long v[10];  // order of RzStats (include/rayz_cuda.h)
};

// Everything a path kernel needs, passed by value (fits the 4 KB parameter space easily).
struct RzPathArgs {
    RzSphereSet set;
    RzMaterials mats;
    RzTextures texs;
    const RzBvhNode *bvh;        // K3 only
    uint32_t bvh_nodes;
    RzCamF32 cam;
    unsigned long long *accum;   // [n_local_px_pad][4] u64 fixed point (2^-32), rgb + sum of Y^2 (only with `moments`)
    unsigned int *unit_counter;  // persistent-kernel work counter (zeroed before launch)
    RzStatsDev *stats;           // STATS builds only
    uint32_t width, height;      // full image
    uint32_t n_local_px;         // pixels owned by this device (compact, band-interleaved rows)
    uint32_t spp, sample_offset, max_depth;
    uint32_t chunk;              // samples per work unit
    uint32_t n_chunks, n_units;
    uint32_t shard_index, shard_count, band_rows;
    uint32_t seed_lo, seed_hi;
    float t_min;
    // K1 staged form.  Queue entries are 4 x float4 (o+time, d+self_k, thr+seg, lp/gpix/sample).
    //   K1a (primary)  : camera segments   -> q_out (+ q_out_keys, the sort key of each surviving ray)
    //   K1c (second)   : q_in through q_in_idx (entries sorted by key) -> second segments -> q_out
    //   K1b (megakern.): q_in -> every later segment, paths regenerated in place
    const float4 *q_in;
    const unsigned int *q_in_count;   // entries in q_in (device counter written by the producing kernel)
    const uint32_t *q_in_idx;         // K1c: entry indices in key order, reach class in the top four bits (RZ_IDX_*)
    const unsigned int *q_in_bins;    // K1c: the sort's scratch words: group ends | units before each group | unit size (RZ_BIN_*)
    unsigned char *bin_lists;         // K1c: per group (cell, direction), the sphere pairs ordered by the smallest reach class that
    uint32_t bin_row;                 //      gets to them (rz_bin_lists_kernel; rows of bin_row bytes, layout: rz_bin_row_bytes)
    float4 *q_out;
    unsigned int *q_out_count;
    unsigned short *q_out_keys;       // 16-bit sort key per appended entry (when a sorted stage follows)
    uint32_t queue_cap;               // entries each queue buffer holds
    uint32_t unit_base;               // first work unit of this pass (primary kernel)
    float focus_dist, lens_radius;    // thin-lens numbers for the tile-frustum cull (derived from the camera)
    float sb_lo[3], sb_hi[3];         // box around every sphere that is not "huge" (radius <= huge_radius: rz_huge_threshold), motion included
    float sb_inv_cell[3];             // cells per unit length along each axis (sort-key cells)
    uint32_t sb_cell_bits[3];         // 9 key bits shared out so that cells come out as cubic as possible
    float huge_radius;                // spheres above this radius lie outside the sphere box: culled by direction only, never by reach
                                      // (the r = 1000 ground, the three r = 1 spheres)
    uint32_t key_sectors;             // direction field of the sort key: 0 = octant (sign of d on each axis), 1 = one of eight 45-degree
                                      // sectors in the plane of the sphere box's two longest axes (key_u, key_w): flat scenes
    uint32_t key_u, key_w;            // those two axes
    float reach_unit;                 // max extent of the box / 32: classes of the sort key's reach field
    unsigned int *err;           // device error word (RZ_DEV_ERR_* bits): set instead of silently dropping work
    uint32_t unit_entries;       // sorted-stage kernels: queue entries per work unit (multiple of 64)
    uint32_t stack_cap;          // K3: usable entries of the per-lane traversal stack (<= RZ_STACK; smaller only in tests)
    const int32_t *self_map;     // K3 fed by a K1 queue: position in the brute-force set -> position in the BVH-ordered set (null: same set)
    uint32_t bvh_active_min;     // K3: lanes that must still be traversing for a burst to go on (ray replacement threshold)
    uint32_t bvh_descend_min;    // K3: a descend round ends once fewer lanes than this are still descending
    uint32_t tile_w;             // K3 camera stage: 0 = a work unit's 32 pixels are consecutive in a row; 8 = an 8 x 4 block (tile lists: the narrower cone)
    uint32_t moments;            // != 0 (RZ_RENDER_MOMENTS): a path that ends in the sky also adds its luminance squared to accum slot 3
    // Adaptive rounds (RZ_RENDER_ADAPTIVE; the LIST instances of the unstaged K3 and of the single-form K1b only): work unit u
    // covers list entries [tile * 32, tile * 32 + 32), and lane k's pixel is px_list[entry] instead of the entry itself.
    const uint32_t *px_list;     // local pixel indices in increasing order (rz_adaptive.cu)
    uint32_t n_list;             // entries in px_list
    uint32_t sobol;              // RZ_SAMPLER_* bits.  != 0 (RZ_RENDER_SOBOL): the launchers run each kernel's SOBOL instance
                                 // (rz_sampler.cuh's pairs), with RZ_SAMPLER_RQMC its SOBOL = 2 instance
};

// RzPathArgs::sobol.  RZ_SAMPLER_RQMC (RZ_RENDER_RQMC) rides in the same word, so that the Philox instances see the very
// arguments they saw before the flag existed; the launchers run the SOBOL = 2 instances for it (rz_pick_sampler): the replicate
// mapping of rz_sobol_pair, and a sky path also adds its clamped luminance to its replicate's sum (rz_rep_offset).
enum { RZ_SAMPLER_SOBOL = 1u, RZ_SAMPLER_RQMC = 2u };
// RZ_RENDER_RQMC's replicate sums share the accumulators' allocation: [n_pad][4] accumulators, then [n_pad][2] replicate sums
// (2^-32 fixed point, slot lp * 2 + (sample & 1)), n_pad = n_local_px rounded up to whole warps.  This is the offset, in words,
// of the replicate sums.
RZ_HD size_t rz_rep_offset(uint32_t n_local_px) { return (size_t)((n_local_px + 31u) / 32u) * 32u * 4u; }

// Guide buffers (rayz_cuda_render_guides, rz_guides_kernel in rz_bvh_trace.cu): the camera segments of a render with these
// RzPathArgs, each followed to its first hit only.  The outputs are the gather root's buffers at the context's rows (peer
// pointers on the other devices), addressed as rz_resolve_kernel addresses its frame.
struct RzGuideArgs {
    RzPathArgs a;                 // set (the BVH-ordered one), mats, texs, bvh, cam, frame and shard fields, spp, sample_offset,
                                  // seeds, t_min, err, stack_cap, bvh_descend_min; nothing else is read
    float4 *out_albedo;           // nullable: rgb = mean first-hit albedo, a = fraction of samples that hit a sphere
    float4 *out_normal;           // nullable: xyz = mean unit normal facing the ray (0 for a miss), w = mean hit distance of the hits
    uint32_t dev_index, dev_count;   // local row lr -> context row ((lr / band_rows) * dev_count + dev_index) * band_rows + lr % band_rows
};

// ---------------------------------------------------------------------------------------------
// Per-pixel noise (RZ_RENDER_MOMENTS, DESIGN.md "Progressive rendering").  Slot 3 of a pixel's accumulator sums Y^2 over its
// paths in the 2^-32 fixed point of slots 0..2, Y = Rec. 709 luminance of the same clamped radiance the three colour atomics
// add.  Paths that end absorbed or at the depth limit add zero to all four slots, as their radiance is zero.
// ---------------------------------------------------------------------------------------------
// Luminance floor of the displayed-value error: the gamma-2 slope 1 / (2 sqrt(Y)) grows without bound at black, where a pixel
// with no variance would otherwise read as 0 / 0.  1e-4 linear is 0.01 displayed, 2.6 steps of 8 bits.
#define RZ_NOISE_Y_FLOOR 1e-4

RZ_HD float rz_clamp_radiance(float v) { return fminf(fmaxf(v, 0.f), 1048576.f); }
// fixed-point sample of a clamped value (the kernels' atomics round to nearest, __float2ull_rn)
RZ_HD unsigned long long rz_fixed32(float v) {
#ifdef __CUDA_ARCH__
    return __float2ull_rn(v * 4294967296.f);
#else
    return (unsigned long long)nearbyint((double)(v * 4294967296.f));
#endif
}
// Y of a path's clamped radiance; the FMAs are explicit so host and device agree bit for bit
RZ_HD float rz_luma(float r, float g, float b) { return fmaf(0.0722f, b, fmaf(0.7152f, g, 0.2126f * r)); }
// Y^2 of a path's clamped radiance, clamped like the colour channels
RZ_HD float rz_luma_sq(float r, float g, float b) {
    const float y = rz_luma(r, g, b);
    return rz_clamp_radiance(y * y);
}

// Standard error of the DISPLAYED value (gamma 2: sqrt of the linear mean, as writePPM shows it) of one pixel from its four
// accumulator slots after n samples, in units of the displayed range [0, 1] (one 8-bit step = 1/255).  f64:
//   Ybar = (0.2126 q0 + 0.7152 q1 + 0.0722 q2) 2^-32 / n,  s^2 = max(0, q3 2^-32 / n - Ybar^2) n / (n - 1),
//   sigma = sqrt(s^2 / n),  e = sigma / (2 sqrt(max(Ybar, RZ_NOISE_Y_FLOOR))).   n < 2 has no variance estimate: +inf.
RZ_HD double rz_pixel_err(unsigned long long q0, unsigned long long q1, unsigned long long q2, unsigned long long q3, uint32_t n) {
    if (n < 2u) return INFINITY;
    const double s = 2.3283064365386962890625e-10, inv = 1.0 / (double)n;   // 2^-32
    const double y = (0.2126 * (double)q0 + 0.7152 * (double)q1 + 0.0722 * (double)q2) * s * inv;
    const double s2 = fmax(0.0, (double)q3 * s * inv - y * y) * ((double)n / (double)(n - 1u));
    return sqrt(s2 * inv) / (2.0 * sqrt(fmax(y, RZ_NOISE_Y_FLOOR)));
}

// RZ_RENDER_RQMC (include/rayz_cuda.h, DESIGN.md "The RQMC estimate"): the error of the iid formula above, scaled by the
// segment's pooled ratio of the two replicates' spread to the iid variance, as it was when the pixel's count was last the frame's
// largest (an adaptive pixel keeps the gain its stopping test read).  A segment is RZ_RQMC_SEGMENT pixels of one row (the
// last of a row may be shorter); local rows are whole global rows, so local pixel lp's segment is a function of (row, x).
#define RZ_RQMC_SEGMENT 64u
RZ_HD uint32_t rz_rqmc_segments(uint32_t width) { return (width + RZ_RQMC_SEGMENT - 1u) / RZ_RQMC_SEGMENT; }
// index of local pixel lp's segment in a [local rows][rz_rqmc_segments(width)] buffer
RZ_HD size_t rz_rqmc_segment_of(uint32_t lp, uint32_t width) {
    const uint32_t lr = lp / width;
    return (size_t)lr * rz_rqmc_segments(width) + (lp - lr * width) / RZ_RQMC_SEGMENT;
}
// V_iid = s^2 / n with rz_pixel_err's s^2; 0 while n < 2
RZ_HD double rz_pixel_var_iid(unsigned long long q0, unsigned long long q1, unsigned long long q2, unsigned long long q3, uint32_t n) {
    if (n < 2u) return 0.0;
    const double s = 2.3283064365386962890625e-10, inv = 1.0 / (double)n;   // 2^-32
    const double y = (0.2126 * (double)q0 + 0.7152 * (double)q1 + 0.0722 * (double)q2) * s * inv;
    return fmax(0.0, (double)q3 * s * inv - y * y) * ((double)n / (double)(n - 1u)) * inv;
}
// V_rep = (mu_0 - mu_1)^2 / 4, mu_r = r_r 2^-32 / (n / 2): the R = 2 replicate variance of the pixel mean; 0 while n < 2
RZ_HD double rz_pixel_var_rep(unsigned long long r0, unsigned long long r1, uint32_t n) {
    if (n < 2u) return 0.0;
    const double inv_m = 2.3283064365386962890625e-10 / (double)(n / 2u);
    const double d = (double)r0 * inv_m - (double)r1 * inv_m;
    return 0.25 * d * d;
}
// G of a segment from its sums of V_rep and V_iid: not clamped; 1 when there is no iid variance to scale
RZ_HD double rz_rqmc_gain(double sum_rep, double sum_iid) { return sum_iid > 0.0 ? sum_rep / sum_iid : 1.0; }
// e = rz_pixel_err * sqrt(G); +inf while n < 2, as rz_pixel_err
RZ_HD double rz_pixel_err_rqmc(unsigned long long q0, unsigned long long q1, unsigned long long q2, unsigned long long q3, uint32_t n,
                               double gain) {
    if (n < 2u) return INFINITY;
    return rz_pixel_err(q0, q1, q2, q3, n) * sqrt(gain);
}
// the error a consumer shows: rz_pixel_err, or under RZ_RENDER_RQMC (gain != null: one gain per local pixel, rz_rqmc_gain_kernel)
// rz_pixel_err_rqmc with local pixel lp's gain
RZ_HD double rz_pixel_err_of(const unsigned long long *q, uint32_t n, const double *gain, uint32_t lp) {
    return gain ? rz_pixel_err_rqmc(q[0], q[1], q[2], q[3], n, gain[lp]) : rz_pixel_err(q[0], q[1], q[2], q[3], n);
}

// writePPM's per-pixel transform (image.zig:35-38) in f64, as the resolve and the denoiser's finish kernel apply it:
// V3.sqrt (x > 0 ? sqrt(x) : 0, vec.zig:87-93) -> clamp(0, 1) -> u8 = trunc(x * 255), into the three bytes of pixel i of out.
RZ_HD void rz_quantise_rgb8(double r, double g, double b, uint8_t *out, size_t i) {
    const double sr = r > 0 ? sqrt(r) : 0, sg = g > 0 ? sqrt(g) : 0, sb = b > 0 ? sqrt(b) : 0;
    const double cr = fmin(fmax(sr, 0.0), 1.0), cg = fmin(fmax(sg, 0.0), 1.0), cb = fmin(fmax(sb, 0.0), 1.0);
    out[i * 3 + 0] = (uint8_t)(cr * 255.0);
    out[i * 3 + 1] = (uint8_t)(cg * 255.0);
    out[i * 3 + 2] = (uint8_t)(cb * 255.0);
}

// ---------------------------------------------------------------------------------------------
// Philox4x32 (Salmon et al., SC'11), seven rounds.  key = 64-bit seed; counter = (global pixel, sample,
// bounce, lane) so the stream is a pure function of WHAT is sampled, never of where it runs:
// any row sharding across GPUs reproduces the full-frame image bit for bit.
// ---------------------------------------------------------------------------------------------
RZ_HD void rz_mulhilo(uint32_t a, uint32_t b, uint32_t &hi, uint32_t &lo) {
#ifdef __CUDA_ARCH__
    hi = __umulhi(a, b);
    lo = a * b;
#else
    const uint64_t p = (uint64_t)a * (uint64_t)b;
    hi = (uint32_t)(p >> 32);
    lo = (uint32_t)p;
#endif
}

// Seven rounds: Philox4x32-7 is the variant Salmon et al. report as already Crush-resistant (BigCrush clean); -10 is their
// default with a safety margin.  Two blocks per camera segment made the ten-round form 16 % of the primary kernel's
// instructions (profiles/r02_primary_kernel_ncu.md).
#define RZ_PHILOX_ROUNDS 7
RZ_HD uint4 rz_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int i = 0; i < RZ_PHILOX_ROUNDS; i++) {
        uint32_t h0, l0, h1, l1;
        rz_mulhilo(0xD2511F53u, c0, h0, l0);
        rz_mulhilo(0xCD9E8D57u, c2, h1, l1);
        const uint32_t n0 = h1 ^ c1 ^ k0;
        const uint32_t n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// 24 random bits -> [0,1)
RZ_HD float rz_u01(uint32_t bits24) { return (float)bits24 * 5.9604644775390625e-8f; }

#include "rz_sampler.cuh"   // RZ_RENDER_SOBOL's pairs

// ---------------------------------------------------------------------------------------------
// small float3 algebra
// ---------------------------------------------------------------------------------------------
RZ_HD float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
RZ_HD float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
RZ_HD float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
RZ_HD float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
RZ_HD float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
RZ_HD float dot3(float3 a, float3 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)); }
RZ_HD float rz_rsqrt(float x) {
#ifdef __CUDA_ARCH__
    return rsqrtf(x);
#else
    return 1.0f / sqrtf(x);
#endif
}
RZ_HD float3 normalize3(float3 a) { return a * rz_rsqrt(dot3(a, a)); }
RZ_HD void rz_sincos2pi(float u, float &s, float &c) {
    // u in [0,1) -> angle in [-pi, pi): keeps the fast-path argument small
    const float a = (u - 0.5f) * 6.283185307179586f;
#ifdef __CUDA_ARCH__
    __sincosf(a, &s, &c);
#else
    s = sinf(a);
    c = cosf(a);
#endif
}

// Uniform direction on the unit sphere from two uniforms.  Same DISTRIBUTION as the
// reference's normalised rejection sample randomUnit (material.zig:196-206); the reference's
// sequential PRNG cannot be matched draw for draw anyway.
RZ_HD float3 rz_uniform_sphere(float u1, float u2) {
    const float z = 1.0f - 2.0f * u1;
    const float r = sqrtf(fmaxf(0.0f, 1.0f - z * z));
    float s, c;
    rz_sincos2pi(u2, s, c);
    return f3(r * c, r * s, z);
}

// ---------------------------------------------------------------------------------------------
// Per-path state
// ---------------------------------------------------------------------------------------------
struct RzRay {
    float3 o, d;   // d is unit length (the reference leaves it un-normalised; geometry is
                   // scale-invariant in d and every consumer normalises or only needs signs)
    float time;
    int self_k;    // sphere (set index) the ray starts on, -1 for camera rays.  Self
                   // re-intersection is resolved analytically instead of by an epsilon:
                   // leaving outward -> cannot re-hit a convex sphere; inward -> far root.
                   // | RZ_SELF_OUT when the scatter step already knows the ray leaves outward.
};
// Flag on RzRay::self_k: the ray leaves its sphere outward by a clear margin (rz_scatter), so the searches skip that sphere
// without testing it.  Equivalent to the arithmetic rule in rz_consider (b < 0 -> rejected), which stays for grazing rays.
#define RZ_SELF_OUT 0x20000000

// ---------------------------------------------------------------------------------------------
// The ray-sphere test every search of the backend uses (packed FP32x2 or scalar, brute force, culled list or BVH leaf):
// Sphere.hitInner (geom.zig:38-58) for a unit-length direction, in the cancellation-free form of Hearn & Baker /
// Ray Tracing Gems ch. 7 (SURVEY section 7):
//     oc = (C - o) + v * time            centre(t) = center.origin + center.dir * ray.time   (geom.zig:40)
//     nb = -(oc . d)                     = -half_b
//     l  = oc + nb * d                   the perpendicular from the centre to the ray's line
//     nd = l . l - r^2                   = -discriminant; the line meets the sphere iff nd < 0
// The textbook discriminant b^2 - (|oc|^2 - r^2) subtracts two numbers of size |oc|^2: 200 units from a sphere of radius 0.2
// its absolute error (~2e-3) is 5 % of r^2.  Here |l| ~ r near the silhouette, so the error stays ~|oc| eps r (1e-4 of r^2 at
// the same distance).  Same instruction count in the packed form (12 FP32x2 per sphere pair against 9 + 2 scalar).
// Every implementation follows THIS operation order per sphere (IEEE rn), so all searches return bit-identical (t, k).
// ---------------------------------------------------------------------------------------------
#define RZ_FAR_BIT 0x40000000

// One row of the per-group sphere lists: u16 end_s[16] | u16 end_m[16] | u16 ls[n_static_pad] | u16 lm[n_pad - n_static_pad] —
// set positions of the stationary / moving spheres in class order; end_x[c] = spheres of classes <= c.
RZ_HD uint32_t rz_bin_row_bytes(uint32_t n_pad) { return (64u + 2u * n_pad + 15u) & ~15u; }

// The sort's output word per slot: queue entry index, with the key's reach class in the top four bits
#define RZ_IDX_MASK 0x0fffffffu
#define RZ_IDX_CLASS_SHIFT 28

// rz_sort.cu's scratch words (one set per side): bins | unit_first | ue
#define RZ_SORT_BINS 4096
#define RZ_BIN_UNIT_FIRST 4096                 /* [4097]: units before each group, then the total */
#define RZ_BIN_UE (4096 + 4097)                /* entries per work unit of this launch */
#define RZ_BIN_SCRATCH_WORDS (4096 + 4097 + 7)

RZ_HD void rz_sphere_test(float cx, float cy, float cz, float vx, float vy, float vz, float w, float ox, float oy, float oz,
                          float dx, float dy, float dz, float time, float &nb, float &nd) {
    const float ocx = fmaf(vx, time, cx - ox), ocy = fmaf(vy, time, cy - oy), ocz = fmaf(vz, time, cz - oz);
    nb = fmaf(ocz, -dz, fmaf(ocy, -dy, ocx * -dx));
    const float lx = fmaf(nb, dx, ocx), ly = fmaf(nb, dy, ocy), lz = fmaf(nb, dz, ocz);
    nd = fmaf(lz, lz, fmaf(ly, ly, fmaf(lx, lx, w)));
}

// A sphere whose line test came out negative (nd < 0).  Root rule of Sphere.hitInner (geom.zig:52-58): the near root if it
// lies in (t_min, best), else the far root.  For the sphere the ray starts on, the t ~ 0 root is excluded analytically
// (RzRay::self_k) instead of by an epsilon.  t_min (default 1e-4) is the FP32 stand-in for renderer.zig:107's 1e-10: a ray
// that starts within t_min of ANOTHER sphere's surface takes that sphere's far root, where the reference would still
// take the near one down to 1e-10 — contact rings ~1e-4 wide around touching spheres (documented deviation).
RZ_HD void rz_consider(int k, float nb, float nd, int self_k, float t_min, float &bt, int &bk) {
    const float sq = sqrtf(-nd);
    const float b = -nb;
    float t = b - sq;
    int tag = k;
    if (k == (self_k & ~RZ_SELF_OUT)) {
        t = (b > 0.0f && !(self_k & RZ_SELF_OUT)) ? b + sq : -1.0f;
        tag = k | RZ_FAR_BIT;
    } else if (t < t_min) {
        t = b + sq;
        tag = k | RZ_FAR_BIT;
    }
    if (t > t_min && t < bt) {
        bt = t;
        bk = tag;
    }
}

// Camera.getRay with rng (camera.zig:59-77) from its five uniforms: jittered pixel position, thin-lens origin on the defocus
// disk, time in [0,1).  Disk sample is polar instead of rejection (same distribution, and area-preserving: strata of (ur, ua)
// stay strata of the disk).
RZ_HD RzRay rz_lens_ray(const RzCamF32 &cam, uint32_t px, uint32_t py, float ux, float uy, float ut, float ur, float ua) {
    const float x = (float)px + (ux - 0.5f);
    const float y = (float)py + (uy - 0.5f);
    RzRay ray;
    ray.o = cam.look_from;
    if (cam.defocus) {
        const float rad = sqrtf(ur);
        float s, c;
        rz_sincos2pi(ua, s, c);
        ray.o = ray.o + cam.defocus_u * (rad * c) + cam.defocus_v * (rad * s);
    }
    const float3 dir = cam.px_du * x + cam.px_dv * y + cam.px_origin - ray.o;
    ray.d = normalize3(dir);
    ray.time = ut;
    ray.self_k = -1;
    return ray;
}

// One Philox block gives the five uniforms: 4 x 24 high bits + 3 x 8 low bits.  With `sobol` != 0 (RZ_RENDER_SOBOL; the kernels
// pass their SOBOL template argument) three Sobol pairs give them instead (rz_sampler.cuh): jitter, lens (radius, angle) and the
// shutter time (first coordinate of the third pair); `sobol` = 2 (RZ_RENDER_RQMC) draws them from the sample's replicate.
RZ_HD RzRay rz_camera_ray(const RzCamF32 &cam, uint32_t px, uint32_t py, uint32_t gpix, uint32_t sample,
                          uint32_t k0, uint32_t k1, int sobol = 0) {
    if (sobol) {
        const bool rqmc = sobol == 2;
        const float2 j = rz_sobol_u01(k0, k1, gpix, RZ_PAIR_CAMERA_JITTER, sample, rqmc);
        const float2 l = rz_sobol_u01(k0, k1, gpix, RZ_PAIR_CAMERA_LENS, sample, rqmc);
        const float t = rz_sobol_u01(k0, k1, gpix, RZ_PAIR_CAMERA_TIME, sample, rqmc).x;
        return rz_lens_ray(cam, px, py, j.x, j.y, t, l.x, l.y);
    }
    const uint4 r = rz_philox(gpix, sample, 0u, 0u, k0, k1);
    const float ux = rz_u01(r.x >> 8), uy = rz_u01(r.y >> 8), ut = rz_u01(r.z >> 8), ur = rz_u01(r.w >> 8);
    const float ua = rz_u01(((r.x & 0xffu) << 16) | ((r.y & 0xffu) << 8) | (r.z & 0xffu));
    return rz_lens_ray(cam, px, py, ux, uy, ut, ur, ua);
}

// Sky of bounceRay's miss branch (renderer.zig:124-125): ((1-t)*1 + (0.5,0.7,1.0)) * t — not a lerp.
RZ_HD float3 rz_sky(float3 d_unit) {
    const float t = 0.5f * (d_unit.y + 1.0f);
    const float a = 1.0f - t;
    return f3((a + 0.5f) * t, (a + 0.7f) * t, (a + 1.0f) * t);
}

// Texture.value (material.zig:44-50) with CheckerTexture's handle recursion (:32-38) unrolled
// into a bounded loop.  The lattice test runs in f64 on the f64-refined hit point: on the
// r=1000 ground sphere |y| is ~1e-8 near the origin, far below FP32 resolution at 1000.
RZ_COLD float3 rz_texture(const RzTextures T, uint32_t tex, double px, double py, double pz) {   // by value: a reference would force the caller's kernel parameters into local memory
#pragma unroll 1
    for (int level = 0; level < 8; level++) {
        if (T.kind[tex] != 0u) break;  // solid
        const double s = T.inv_scale[tex];
        const long long ix = (long long)floor(px * s);
        const long long iy = (long long)floor(py * s);
        const long long iz = (long long)floor(pz * s);
        const long long m = (ix + iy + iz) & 1ll;  // floor-mod 2 (two's complement)
        tex = (m == 0) ? T.even[tex] : T.odd[tex];
    }
    const float4 c = T.color[tex];
    return f3(c.x, c.y, c.z);
}

// The one-level case of rz_texture with its operands already in registers (RzMaterials::rec): the same f64 lattice test.
RZ_HD float3 rz_checker2(const RzMatRec &M, double px, double py, double pz) {
    const long long ix = (long long)floor(px * M.inv_scale), iy = (long long)floor(py * M.inv_scale), iz = (long long)floor(pz * M.inv_scale);
    return ((ix + iy + iz) & 1ll) == 0 ? M.color : M.odd;
}

struct RzHit {
    double px, py, pz;  // hit point, f64
    float3 p;           // same, rounded: next ray origin
    float3 n;           // shading normal, flipped against the ray (Hit.init, hit.zig:33-37)
    bool front;
};

// Re-evaluate the winning sphere in f64 from the FP32 ray (Sphere.hitInner, geom.zig:38-66, with
// the root the FP32 search selected).  ~40 DFMA-class ops once per segment vs ~6000 FP32
// instructions of brute-force search; it makes point/normal self-consistent to 1e-13 so the
// self-intersection rule and the checker lattice are exact.
RZ_HD RzHit rz_refine_hit(const RzSphereSet &S, const RzRay &ray, int k, bool far_root) {
    const double4 c = S.c64[k];
    const double4 v = S.v64[k];
    const double tm = (double)ray.time;
    const double cx = fma(v.x, tm, c.x), cy = fma(v.y, tm, c.y), cz = fma(v.z, tm, c.z);
    const double ox = ray.o.x, oy = ray.o.y, oz = ray.o.z;
    const double dx = ray.d.x, dy = ray.d.y, dz = ray.d.z;
    const double ocx = cx - ox, ocy = cy - oy, ocz = cz - oz;
    const double a = dx * dx + dy * dy + dz * dz;
    const double hb = dx * ocx + dy * ocy + dz * ocz;
    const double cc = (ocx * ocx + ocy * ocy + ocz * ocz) - c.w * c.w;
    double disc = hb * hb - a * cc;
    if (!(disc > 0.0)) disc = 0.0;  // FP32 said "grazing hit"; f64 says tangent/miss: clamp
    const double rt = sqrt(disc);
    // 1 / a without an f64 division (38 instructions): d is unit length to FP32 rounding, a = 1 + e with |e| ~ 1e-7, so
    // x0 = 2 - a is off by e^2 ~ 1e-14 and one Newton step leaves e^4
    const double x0 = 2.0 - a;
    const double inv_a = x0 * (2.0 - a * x0);
    const double t = (far_root ? (hb + rt) : (hb - rt)) * inv_a;
    RzHit h;
    h.px = fma(dx, t, ox);
    h.py = fma(dy, t, oy);
    h.pz = fma(dz, t, oz);
    const double inv_r = v.w;   // 1 / radius, divided once at upload (RzSphereSet::v64)
    double nx = (h.px - cx) * inv_r, ny = (h.py - cy) * inv_r, nz = (h.pz - cz) * inv_r;
    h.front = (nx * dx + ny * dy + nz * dz) < 0.0;
    if (!h.front) { nx = -nx; ny = -ny; nz = -nz; }
    h.n = f3((float)nx, (float)ny, (float)nz);
    h.p = f3((float)h.px, (float)h.py, (float)h.pz);
    return h;
}

// material.zig:179-183; pow(1-cos,5) as repeated multiplication
RZ_HD float rz_reflectance(float cosv, float ri) {
    float r0 = (1.0f - ri) / (1.0f + ri);
    r0 *= r0;
    const float m = 1.0f - cosv;
    const float m2 = m * m;
    return r0 + (1.0f - r0) * (m2 * m2 * m);
}

// DiffuseScatterMethod.UNIT_SPHERE: normal + point in ball; UNIT_SPHERE_SURFACE: normal + unit vector (material.zig:78-82).
// No reference scene selects them (default HEMISPHERE, :74): out of line.
RZ_COLD float3 rz_diffuse_other(uint32_t method, float3 s, float3 n, float uz) {
    const float rad = (method == 0u) ? cbrtf(uz) : 1.0f;
    float3 t = n + s * rad;
    if (dot3(t, t) < 1e-12f) t = n;
    return normalize3(t);
}

// Material.scatter (material.zig:167-176).  Returns false when the path is absorbed
// (MetallicMaterial.scatter -> null, :116-117).  `ray` is replaced by the scattered ray,
// `att` receives the attenuation.  u = four uniforms of this bounce's Philox block.
RZ_HD bool rz_scatter(const RzMatRec &M, const RzTextures &T, const RzHit &h, int k, float4 u, RzRay &ray, float3 &att) {
    const uint32_t kind = M.kind;
    float3 nd;
    if (kind == 0u) {
        // DiffuseMaterial.scatter (:77-101).  HEMISPHERE (default, :74): direction of a uniform
        // ball sample flipped into the normal's hemisphere == uniform over the hemisphere,
        // no cosine weighting, attenuation = albedo.
        const uint32_t method = M.method;
        const float3 s = rz_uniform_sphere(u.x, u.y);
        if (method == 2u) nd = dot3(s, h.n) > 0.0f ? s : s * -1.0f;
        else nd = rz_diffuse_other(method, s, h.n, u.z);
        att = M.solid ? M.color : M.checker2 ? rz_checker2(M, h.px, h.py, h.pz) : rz_texture(T, M.tex, h.px, h.py, h.pz);
    } else if (kind == 1u) {
        // MetallicMaterial.scatter (:108-131): unit mirror direction + min(fuzz,1) * unit vector
        const float dn = dot3(ray.d, h.n);
        float3 r = ray.d - h.n * (2.0f * dn);
        const float fuzz = M.fuzz;
        if (fuzz > 0.0f) r = r + rz_uniform_sphere(u.x, u.y) * fminf(fuzz, 1.0f);
        if (!(dot3(r, h.n) > 0.0f)) return false;
        nd = normalize3(r);
        att = M.solid ? M.color : M.checker2 ? rz_checker2(M, h.px, h.py, h.pz) : rz_texture(T, M.tex, h.px, h.py, h.pz);
    } else {
        // DielectricMaterial.scatter (:137-159).  The reference leaves cos/sin/sqrt unclamped
        // (NaN on rounding, mapped to 0 at output by V3.sqrt); FP32 clamps to stay NaN-free.
        const float ior = M.ior;
        const float eta = h.front ? 1.0f / ior : ior;
        const float cos_t = fminf(-dot3(ray.d, h.n), 1.0f);
        const float sin_t = sqrtf(fmaxf(0.0f, 1.0f - cos_t * cos_t));
        if (eta * sin_t > 1.0f || rz_reflectance(cos_t, eta) > u.x) {
            nd = ray.d - h.n * (2.0f * dot3(ray.d, h.n));       // reflect (:185-187)
        } else {
            const float3 perp = (ray.d + h.n * cos_t) * eta;    // refract (:189-194)
            const float par = -sqrtf(fmaxf(0.0f, 1.0f - dot3(perp, perp)));
            nd = perp + h.n * par;
        }
        nd = normalize3(nd);
        att = f3(1.0f, 1.0f, 1.0f);
    }
    ray.o = h.p;
    ray.d = nd;
    // outward by a margin far above the FP32 error of b = (C - o).d (|C - o| 2^-22: r = 1000 -> 2e-4 r): b < 0 for certain
    const float out = dot3(nd, h.n);
    ray.self_k = ((h.front ? out : -out) > 1e-3f) ? (k | RZ_SELF_OUT) : k;   // time is kept (material.zig:92,122,155)
    return true;
}

// local (compact, band-interleaved) pixel index -> global pixel coordinates
RZ_HD void rz_local_to_global(uint32_t lp, uint32_t width, uint32_t shard_index, uint32_t shard_count,
                              uint32_t band_rows, uint32_t &i, uint32_t &j) {
    const uint32_t lr = lp / width;
    i = lp - lr * width;
    if (shard_count <= 1u) { j = lr; return; }
    const uint32_t lb = lr / band_rows;
    const uint32_t within = lr - lb * band_rows;
    j = (lb * shard_count + shard_index) * band_rows + within;
}

// ---------------------------------------------------------------------------------------------
// Sort key of the staged K1's queues, and its decoder.  Host + device: tests/hostsim checks on the CPU
// that the bounds rz_key_bounds derives from a key contain every ray rz_sort_key maps to that key.
// ---------------------------------------------------------------------------------------------
// When does a ray leave the box around all non-huge spheres for good?  (<= 0: it never enters it.)
RZ_HD float rz_box_exit(const RzPathArgs &a, const RzRay &ray) {
    float t = 3.0e38f;
    const float o[3] = {ray.o.x, ray.o.y, ray.o.z}, d[3] = {ray.d.x, ray.d.y, ray.d.z};
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {   // one division per axis, no branches: the face the ray heads for
        float ta = ((d[ax] < 0.f ? a.sb_lo[ax] : a.sb_hi[ax]) - o[ax]) / d[ax];
        if (d[ax] == 0.f) ta = (o[ax] < a.sb_lo[ax] || o[ax] > a.sb_hi[ax]) ? 0.f : 3.0e38f;   // parallel to the slab: outside for ever, or never leaves
        t = fminf(t, ta);
    }
    return t;
}

RZ_HD int rz_clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Host side: the key's grid over the box [lo, hi] around the non-huge spheres.  `cell_bits` key bits (<= 9) are shared out
// over the axes — each bit halves the cells of the axis whose cells are currently largest, so cells come out as cubic as
// the extents allow; reach classes are measured in units of 1/32 of the longest extent.
RZ_HD float rz_pick3(float x, float y, float z, uint32_t ax) { return ax == 0u ? x : ax == 1u ? y : z; }

// Which spheres stay OUTSIDE the sphere box ("huge": tested by every ray whose direction field can reach them, whatever its
// reach class): those above 4 x the median radius — in the reference scenes the r = 1000 ground and the three r = 1 spheres,
// which would otherwise make the box 2.0 high instead of 0.9 and more than double how long an upward ray counts as inside
// it — but never more than max(4, n / 32) of them, largest first (each costs every list a test).  Returns the largest
// radius that still belongs INSIDE the box.  Host only.
inline double rz_huge_threshold(const double *radius, uint32_t n, double factor = 4.0) {
    if (n == 0u) return 3.0e38;
    std::vector<double> r(radius, radius + n);
    std::nth_element(r.begin(), r.begin() + n / 2, r.end());
    double thr = factor * r[n / 2];
    const uint32_t cap = n / 32u > 4u ? n / 32u : 4u;
    if (n > cap) {   // more than `cap` above the threshold: only the cap largest stay outside
        std::nth_element(r.begin(), r.begin() + (n - 1u - cap), r.end());
        if (r[n - 1u - cap] > thr) thr = r[n - 1u - cap];
    }
    return thr;
}

// key_mode: 0 = octant direction field, 1 = sectors, -1 = by the shape of the box (sectors when it is flat: the third
// extent under 0.35 of the other two, so that almost every long ray travels near the plane of the two long axes).
inline void rz_key_grid(RzPathArgs &a, const float (&lo)[3], const float (&hi)[3], int cell_bits, int key_mode = -1) {
    float ext = 0.f, e3[3];
    uint32_t bits[3] = {0, 0, 0};
    for (int ax = 0; ax < 3; ax++) {
        a.sb_lo[ax] = lo[ax]; a.sb_hi[ax] = hi[ax];
        e3[ax] = hi[ax] - lo[ax];
        if (!(e3[ax] > 0.f) || !(e3[ax] < 1.0e30f)) e3[ax] = 0.f;
        ext = e3[ax] > ext ? e3[ax] : ext;
    }
    int hax = 0;
    for (int ax = 1; ax < 3; ax++) if (e3[ax] < e3[hax]) hax = ax;
    a.key_u = (uint32_t)((hax + 1) % 3); a.key_w = (uint32_t)((hax + 2) % 3);
    if (a.key_u > a.key_w) { const uint32_t t = a.key_u; a.key_u = a.key_w; a.key_w = t; }
    const float e_min2 = e3[a.key_u] < e3[a.key_w] ? e3[a.key_u] : e3[a.key_w];
    const bool flat = e_min2 > 0.f && e3[hax] < 0.35f * e_min2;
    a.key_sectors = key_mode < 0 ? (flat ? 1u : 0u) : (uint32_t)(key_mode > 2 ? 1 : key_mode);
    if (a.key_sectors == 2u && cell_bits > 8) cell_bits = 8;   // 16 sectors take a bit of the 12 the groups are made of
    // with sector keys every cell bit goes to the two long axes: the cull is a wedge in their plane, and a flat box has
    // next to no origins in its upper half anyway
    float w3[3] = {e3[0], e3[1], e3[2]};
    if (a.key_sectors) w3[hax] = 0.f;
    for (int b = 0; b < cell_bits; b++) {
        int best = 0;
        for (int ax = 1; ax < 3; ax++)
            if (w3[ax] / (float)(1u << bits[ax]) > w3[best] / (float)(1u << bits[best])) best = ax;
        bits[best]++;
    }
    for (int ax = 0; ax < 3; ax++) {
        a.sb_cell_bits[ax] = bits[ax];
        a.sb_inv_cell[ax] = e3[ax] > 0.f ? (float)(1u << bits[ax]) / e3[ax] : 0.f;
    }
    a.reach_unit = ext > 0.f ? ext / 32.0f : 1.0f;
}

#define RZ_TAN_22_5 0.41421356f
// bits of the key's direction field: 3 (octants, eight 45-degree sectors) or 4 (sixteen 22.5-degree sectors)
RZ_HD uint32_t rz_key_dir_bits(const RzPathArgs &a) { return a.key_sectors == 2u ? 4u : 3u; }

// Sort key of a scattered ray: [origin cell 9 bits][direction 3 bits][reach class 4 bits] = 16 bits (or [8][4][4]).  Rays with equal keys
// start in the same cell of the sphere box (the 9 bits are shared out over the axes by extent), head the same way — the same
// octant, or for a flat sphere box the same 45-degree sector in the plane of its two long axes (rz_key_grid) — and stay
// inside the sphere box for a similar distance: which is what the sorted-segment kernel's per-group lists feed on.
RZ_HD uint32_t rz_sort_key(const RzPathArgs &a, const RzRay &ray) {
    const int nx = (1 << a.sb_cell_bits[0]) - 1, ny = (1 << a.sb_cell_bits[1]) - 1, nz = (1 << a.sb_cell_bits[2]) - 1;
    const int cx = rz_clampi((int)((ray.o.x - a.sb_lo[0]) * a.sb_inv_cell[0]), 0, nx);
    const int cy = rz_clampi((int)((ray.o.y - a.sb_lo[1]) * a.sb_inv_cell[1]), 0, ny);
    const int cz = rz_clampi((int)((ray.o.z - a.sb_lo[2]) * a.sb_inv_cell[2]), 0, nz);
    const uint32_t cell = (uint32_t)(((cx << a.sb_cell_bits[1]) | cy) << a.sb_cell_bits[2]) | (uint32_t)cz;   // 9 bits
    uint32_t oct;
    float te = rz_box_exit(a, ray);
    if (a.key_sectors) {   // sector of the direction's projection on the (u, w) plane: signs of d_u, d_w and which of the two is larger
        const float du = rz_pick3(ray.d.x, ray.d.y, ray.d.z, a.key_u), dw = rz_pick3(ray.d.x, ray.d.y, ray.d.z, a.key_w);
        const float mu = fabsf(du), mw = fabsf(dw);
        // sector keys put every cell bit into the (u, w) plane and cull in that plane only (the third axis of the box of origins is
        // open-ended): what counts is how far the ray gets IN THE PLANE before it leaves the sphere box — a ray that climbs
        // steeply out of a flat box leaves it after a short stretch of ground
        te *= fminf(sqrtf(fmaf(du, du, dw * dw)) * 1.0001f, 1.0f);
        oct = (du < 0.f ? 1u : 0u) | (dw < 0.f ? 2u : 0u) | (mu < mw ? 4u : 0u);
        // 16 sectors: + which half of the 45-degree wedge, the one next to the larger component's axis (bit set) or the diagonal's
        if (a.key_sectors == 2u) oct |= fminf(mu, mw) < RZ_TAN_22_5 * fmaxf(mu, mw) ? 8u : 0u;
    } else {
        oct = (ray.d.x < 0.f ? 1u : 0u) | (ray.d.y < 0.f ? 2u : 0u) | (ray.d.z < 0.f ? 4u : 0u);
    }
    // 16 reach classes, two per octave of te / reach_unit from 1/4 up
#ifdef __CUDA_ARCH__
    const float l2 = __log2f(fmaxf(te / a.reach_unit, 0.25f));
#else
    const float l2 = log2f(fmaxf(te / a.reach_unit, 0.25f));
#endif
    const int reach = rz_clampi((int)(2.0f * l2 + 4.0f), 0, 15);
    return (((cell << rz_key_dir_bits(a)) | oct) << 4) | (uint32_t)reach;
}

// What a key says about its rays, conservatively: the origin lies in [lo, hi] (the key's cell, open-ended for the outermost
// cells, where out-of-box origins are clamped), the direction's signs are `oct` (bit set <=> component < 0), and the ray
// leaves the sphere box before T (the upper edge of the reach class; the top class is unbounded).
RZ_HD void rz_key_bounds(const RzPathArgs &a, uint32_t key, float (&lo)[3], float (&hi)[3], uint32_t &oct, float &T) {
    const int nbx = (int)a.sb_cell_bits[0], nby = (int)a.sb_cell_bits[1], nbz = (int)a.sb_cell_bits[2];
    const int reach = (int)(key & 15u);
    const uint32_t db = rz_key_dir_bits(a);
    oct = (key >> 4) & ((1u << db) - 1u);
    const uint32_t cell = key >> (4u + db);
    const int c3[3] = {(int)(cell >> (nby + nbz)), (int)((cell >> nbz) & ((1u << nby) - 1u)), (int)(cell & ((1u << nbz) - 1u))};
    const int n3[3] = {(1 << nbx) - 1, (1 << nby) - 1, (1 << nbz) - 1};
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {
        const float w = a.sb_inv_cell[ax] > 0.f ? 1.0f / a.sb_inv_cell[ax] : 3.0e38f;   // cell width
        lo[ax] = c3[ax] <= 0 ? -3.0e38f : fmaf((float)c3[ax], w, a.sb_lo[ax]) - 1e-4f * w;
        hi[ax] = c3[ax] >= n3[ax] ? 3.0e38f : fmaf((float)(c3[ax] + 1), w, a.sb_lo[ax]) + 1e-4f * w;
    }
    // class c holds te / reach_unit in [2^((c-4)/2), 2^((c-3)/2)); class 15 is open-ended
    T = reach >= 15 ? 3.0e38f : a.reach_unit * exp2f(0.5f * (float)(reach - 3)) * 1.0001f;
}

// ---------------------------------------------------------------------------------------------
// The two culls of the staged K1, as host + device functions (tests/hostsim checks on the CPU that neither ever drops a
// sphere one of its rays hits).  A sphere enters as its packed operands: centre at shutter time 0, velocity, w = -r^2.
// ---------------------------------------------------------------------------------------------
// Primary kernel: cone around the camera rays of a 32-pixel tile.
struct RzTileCone {
    float3 apex, ax;     // lens centre; unit axis = normalised sum of the tile's unit pixel directions
    float tan_t;         // tangent of the half-angle (to the farthest pixel corner), with margin
    float inv_f;         // 1 / (0.9 focus distance): growth of the thin-lens blur beyond the focus plane
    float lens_radius;
    bool cull;           // false: very wide tiles (tiny images) test everything
};

// direction from the lens centre to the centre of pixel (pi, pj) on the focus plane (not normalised)
RZ_HD float3 rz_tile_pixel_dir(const RzCamF32 &cam, uint32_t pi, uint32_t pj) {
    return cam.px_origin + cam.px_du * (float)pi + cam.px_dv * (float)pj - cam.look_from;
}

// smallest cosine between the axis and the four corners of the pixel whose centre direction is pc
RZ_HD float rz_tile_corner_cos(const RzCamF32 &cam, float3 pc, float3 ax) {
    float cmin = 1.0f;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const float3 q = pc + cam.px_du * ((c & 1) ? 0.5f : -0.5f) + cam.px_dv * ((c & 2) ? 0.5f : -0.5f);
        cmin = fminf(cmin, dot3(ax, normalize3(q)));
    }
    return cmin;
}

// ax_sum: sum of the valid pixels' unit directions; normalises it and returns false if the tile has no direction
RZ_HD bool rz_tile_axis(float3 &ax_sum) {
    const float al = dot3(ax_sum, ax_sum);
    ax_sum = al > 1e-12f ? ax_sum * rz_rsqrt(al) : f3(0.f, 0.f, 1.f);
    return al > 1e-12f;
}

RZ_HD RzTileCone rz_tile_cone(const RzCamF32 &cam, float3 ax, bool has_axis, float cmin, float focus_dist, float lens_radius) {
    RzTileCone C;
    C.apex = cam.look_from;
    C.ax = ax;
    C.cull = cmin > 0.2f && has_axis;
    C.tan_t = C.cull ? sqrtf(fmaxf(0.f, 1.f - cmin * cmin)) / cmin * 1.05f + 1e-4f : 0.f;
    C.inv_f = 1.0f / fmaxf(0.9f * focus_dist, 1e-6f);
    C.lens_radius = lens_radius;
    return C;
}

RZ_HD bool rz_tile_keep(const RzTileCone &C, float cx, float cy, float cz, float vx, float vy, float vz, float w) {
    if (!(w < 0.f)) return false;                         // padding entry (-r^2 = +1)
    if (!C.cull) return true;
    const float vl = sqrtf(vx * vx + vy * vy + vz * vz);
    const float re = sqrtf(-w) + 0.5f * vl;               // sphere swept over time in [0,1): midpoint + half the travel
    const float3 vv = f3(fmaf(0.5f, vx, cx), fmaf(0.5f, vy, cy), fmaf(0.5f, vz, cz)) - C.apex;
    const float h = dot3(vv, C.ax), d2 = dot3(vv, vv);
    const float smax = fmaxf(h + re, 0.f);                // farthest along-axis extent of the sphere
    // cone radius there + thin-lens blur (grows beyond the focus plane) + margins for FP32 and the 1.05 above
    const float rad = re * 1.02f + 0.02f + C.lens_radius * (1.f + smax * C.inv_f) + smax * C.tan_t;
    if (d2 <= rad * rad) return true;                     // apex inside / next to the sphere
    if (h + re < 0.f) return false;                       // entirely behind the camera
    return fmaxf(d2 - h * h, 0.f) <= rad * rad;
}

// K3's camera stage culls a TREE against the cone: a child box enters as its bounding sphere (centre, half diagonal with a margin
// for the FP32 evaluation), stationary.  Every sphere inside the box — swept over the shutter: the builders' boxes cover both
// ends — lies inside that bounding sphere, and rz_tile_keep only grows more permissive with the radius at a centre at most that
// radius away, so a box is never dropped while a sphere inside it would be kept (tests/hostsim checks it on the CPU).
RZ_HD bool rz_tile_keep_box(const RzTileCone &C, float lox, float hix, float loy, float hiy, float loz, float hiz) {
    const float ex = hix - lox, ey = hiy - loy, ez = hiz - loz;
    const float r2 = 0.25f * (ex * ex + ey * ey + ez * ez) * 1.0002f + 1e-12f;
    return rz_tile_keep(C, 0.5f * (lox + hix), 0.5f * (loy + hiy), 0.5f * (loz + hiz), 0.f, 0.f, 0.f, -r2);
}

// Sorted-stage kernel: what the rays of one unit have in common, merged from the bounds of their keys (rz_key_bounds).
struct RzUnitBounds {
    float lo[3], hi[3];          // box of the origins
    float T;                     // longest stay inside the sphere box
    unsigned all_pos, all_neg;   // octant keys: bit ax set: every ray has d[ax] >= 0 / d[ax] < 0
    unsigned sectors;            // sector keys: bit s set: some ray's direction lies in sector s
};

RZ_HD void rz_unit_bounds_init(RzUnitBounds &U) {
    for (int ax = 0; ax < 3; ax++) { U.lo[ax] = 3.0e38f; U.hi[ax] = -3.0e38f; }
    U.T = 0.f; U.all_pos = 7u; U.all_neg = 7u; U.sectors = 0u;
}

// Upper edge of reach class c (what rz_key_bounds returns as T), with the margin for the FP32 evaluation of the exits that
// rz_unit_bounds_finish applies.  Class 15 is open-ended.
RZ_HD float rz_class_T(const RzPathArgs &a, int c) {
    return c >= 15 ? 3.0e38f : fminf(a.reach_unit * exp2f(0.5f * (float)(c - 3)) * 1.0001f, 1.0e30f) * 1.001f;
}

RZ_HD void rz_unit_bounds_add_key(RzUnitBounds &U, const RzPathArgs &a, uint32_t key) {
    float lo[3], hi[3], Tk;
    uint32_t oct;
    rz_key_bounds(a, key, lo, hi, oct, Tk);
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {
        U.lo[ax] = fminf(U.lo[ax], lo[ax]);
        U.hi[ax] = fmaxf(U.hi[ax], hi[ax]);
        if ((oct >> ax) & 1u) U.all_pos &= ~(1u << ax); else U.all_neg &= ~(1u << ax);   // key bit set <=> d < 0
    }
    U.sectors |= 1u << oct;
    U.T = fmaxf(U.T, Tk);
}

// after the merge over the unit: +inf-safe, with margin for the FP32 evaluation of the exits
RZ_HD void rz_unit_bounds_finish(RzUnitBounds &U) { U.T = fminf(U.T, 1.0e30f) * 1.001f; }

// Can a ray of the unit reach the sphere at all, whatever its reach?  false: behind the cell box on an axis along which every
// ray of the unit moves the other way, or outside the unit's direction wedge (or a padding entry).  d2 = squared distance from
// the box of the origins to the segment the sphere's centre travels over the shutter interval (per axis: to its bounding
// interval), re = its radius with margins.  Huge spheres: d2 = 0, re = 0 (every reach class).
// Sector keys: can a ray whose direction projects into sector s of the (u, w) plane get from the box of origins to the sphere?
// Sector s = (d_u < 0, d_w < 0, |d_u| < |d_w|) is the wedge {n1.d >= 0, n2.d >= 0}: n1 along one axis, n2 a diagonal.  A point
// p is reached from an origin o with such a direction only if n.(p - o) >= 0 for both; for a sphere, >= -|n| re; over the box,
// n.o is replaced by its minimum (each half-plane with its own best corner: conservative).
RZ_HD bool rz_sector_reaches(float lo_u, float hi_u, float lo_w, float hi_w, uint32_t s, float cu, float cw, float cu1, float cw1, float re,
                             bool sixteen = false) {
    const float au = (s & 1u) ? -1.f : 1.f, aw = (s & 2u) ? -1.f : 1.f;   // |d_u| = au d_u, |d_w| = aw d_w
    const bool w_larger = (s & 4u) != 0u;
    // In folded coordinates (M = the larger component's axis, m = the smaller's, both made positive) the sector is the wedge of
    // polar angles [p_lo, p_hi]: 8 sectors: [0, 45]; 16 sectors: [0, 22.5] (bit 3 set) or [22.5, 45].  Inward unit normals:
    // n_lo = (-sin p_lo, cos p_lo), n_hi = (sin p_hi, -cos p_hi).
    const bool near_axis = !sixteen || (s & 8u) != 0u, near_diag = !sixteen || (s & 8u) == 0u;
    const float loM = near_axis ? 0.f : -0.38268343f, lom = near_axis ? 1.f : 0.92387953f;
    const float hiM = near_diag ? 0.70710678f : 0.38268343f, him = near_diag ? -0.70710678f : -0.92387953f;
    // back to (u, w): M is w when w is the larger one; each axis with its sign
    const float n1u = (w_larger ? lom : loM) * au, n1w = (w_larger ? loM : lom) * aw;
    const float n2u = (w_larger ? him : hiM) * au, n2w = (w_larger ? hiM : him) * aw;
    auto box_min = [&](float nu, float nw) {   // min over the box of n.o (the box may be open-ended: +-3e38 times 0 stays 0)
        return (nu > 0.f ? lo_u : hi_u) * nu + (nw > 0.f ? lo_w : hi_w) * nw;
    };
    const float rem = re * 1.0001f + 1e-5f;   // the normals are unit length to FP32 rounding
    // (cu, cw) -> (cu1, cw1): the segment the sphere's centre travels; a half-plane drops it only if it drops both ends
    if (fmaxf(n1u * cu + n1w * cw, n1u * cu1 + n1w * cw1) + rem < box_min(n1u, n1w)) return false;
    if (fmaxf(n2u * cu + n2w * cw, n2u * cu1 + n2w * cw1) + rem < box_min(n2u, n2w)) return false;
    return true;
}

RZ_HD bool rz_unit_reachable(const RzUnitBounds &U, const RzPathArgs &a, float cx, float cy, float cz, float vx, float vy, float vz, float w,
                             float &d2, float &re) {
    d2 = 0.f; re = 0.f;
    if (!(w < 0.f)) return false;                                  // padding entry
    const float r = sqrtf(-w);
    const bool huge = r > a.huge_radius;                           // outside the sphere box: never culled by distance, only by direction
    re = r * 1.02f + 0.02f;                                        // radius + margin
    // over the shutter interval the centre travels the segment c0 -> c0 + v (geom.zig:40, time in [0, 1)): every test below is
    // made against the whole segment — its bounding interval per axis, its better end per half-plane — not against a sphere
    // around the midpoint blown up by half the travel (the reference scenes' movers only bounce vertically: r + 0.25 -> r)
    const float c0[3] = {cx, cy, cz}, c1[3] = {cx + vx, cy + vy, cz + vz};
    if (a.key_sectors) {
        bool any = false;
        const float lo_u = rz_pick3(U.lo[0], U.lo[1], U.lo[2], a.key_u), hi_u = rz_pick3(U.hi[0], U.hi[1], U.hi[2], a.key_u);
        const float lo_w = rz_pick3(U.lo[0], U.lo[1], U.lo[2], a.key_w), hi_w = rz_pick3(U.hi[0], U.hi[1], U.hi[2], a.key_w);
        const float cu0 = rz_pick3(c0[0], c0[1], c0[2], a.key_u), cw0 = rz_pick3(c0[0], c0[1], c0[2], a.key_w);
        const float cu1 = rz_pick3(c1[0], c1[1], c1[2], a.key_u), cw1 = rz_pick3(c1[0], c1[1], c1[2], a.key_w);
        for (unsigned m = U.sectors; m && !any; m &= m - 1u) {
#ifdef __CUDA_ARCH__
            const uint32_t s = (uint32_t)__ffs((int)m) - 1u;
#else
            uint32_t s = 0; while (!((m >> s) & 1u)) s++;
#endif
            any = rz_sector_reaches(lo_u, hi_u, lo_w, hi_w, s, cu0, cw0, cu1, cw1, re, a.key_sectors == 2u);
        }
        if (!any) return false;
    }
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {
        const float smin = fminf(c0[ax], c1[ax]), smax = fmaxf(c0[ax], c1[ax]);
        if (!a.key_sectors) {
            if (((U.all_pos >> ax) & 1u) && smax + re < U.lo[ax]) return false;   // every ray moves up this axis: sphere is behind
            if (((U.all_neg >> ax) & 1u) && smin - re > U.hi[ax]) return false;
        }
        const float dd = fmaxf(0.f, fmaxf(U.lo[ax] - smax, smin - U.hi[ax]));
        d2 = fmaf(dd, dd, d2);
    }
    if (huge) { d2 = 0.f; re = 0.f; }                              // a ray can meet it after it has left the sphere box: every reach class
    return true;
}

RZ_HD bool rz_unit_keep(const RzUnitBounds &U, const RzPathArgs &a, float cx, float cy, float cz, float vx, float vy, float vz, float w) {
    float d2, re;
    if (!rz_unit_reachable(U, a, cx, cy, cz, vx, vy, vz, w, d2, re)) return false;
    const float rad = U.T + re;
    return d2 <= rad * rad;                                        // within reach of some ray of the unit
}

// The SMALLEST reach class whose rays can reach the sphere from the unit's box (16: none can).  A ray of class c stays inside
// the sphere box for less than rz_class_T(c), so it needs exactly the spheres of classes <= c: the sorted-stage kernel orders
// its sphere list by this number and gives every batch of rays the prefix that belongs to the batch's largest class.
// Monotone in c by construction: the answer is found from a log2 estimate and then corrected with the predicate of
// rz_unit_keep itself in both directions, so it never errs on the side of dropping a sphere.
RZ_HD int rz_unit_class(const RzUnitBounds &U, const RzPathArgs &a, float cx, float cy, float cz, float vx, float vy, float vz, float w) {
    float d2, re;
    if (!rz_unit_reachable(U, a, cx, cy, cz, vx, vy, vz, w, d2, re)) return 16;
    auto within = [&](int c) { const float rad = rz_class_T(a, c) + re; return d2 <= rad * rad; };
    const float dist = sqrtf(d2) - re;
    if (!(dist > 0.f)) return 0;
#ifdef __CUDA_ARCH__
    const float l2 = __log2f(dist / a.reach_unit);
#else
    const float l2 = log2f(dist / a.reach_unit);
#endif
    int c = rz_clampi((int)(2.0f * l2 + 3.0f), 0, 15);
    while (c > 0 && within(c - 1)) c--;
    while (c < 15 && !within(c)) c++;
    return c;
}

// the unit's box of origins and common direction signs from one key's cell and octant (the reach class is handled per ray)
RZ_HD void rz_unit_bounds_add_cell(RzUnitBounds &U, const RzPathArgs &a, uint32_t key) {
    float lo[3], hi[3], Tk;
    uint32_t oct;
    rz_key_bounds(a, key, lo, hi, oct, Tk);
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {
        U.lo[ax] = fminf(U.lo[ax], lo[ax]);
        U.hi[ax] = fmaxf(U.hi[ax], hi[ax]);
        if ((oct >> ax) & 1u) U.all_pos &= ~(1u << ax); else U.all_neg &= ~(1u << ax);
    }
    U.sectors |= 1u << oct;
}
