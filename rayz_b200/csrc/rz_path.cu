// rz_path.cu — K1: the brute-force FP32 path tracer for sm_100a, three kernels and a table builder.
//
// Replaces the body of Tracer.render's pixel loop and everything under it
// (reference src/renderer.zig:85-96, bounceRay :103-126, BVH.findHit hit.zig:181-216,
// Sphere.hitInner geom.zig:38-66, Material.scatter material.zig:167-176).
//
//   rz_primary_kernel  (K1a)  camera segments; sphere set culled against each 32-pixel tile's frustum
//   rz_second_kernel   (K1c)  the next few segments, one per launch, over queue entries grouped by (origin cell, direction);
//                             a work unit's rays share one group and search that group's precomputed sphere list
//   rz_bin_lists_kernel       those lists: per group, the spheres its rays can reach, ordered by reach class
//   rz_path_kernel     (K1b)  the whole path loop in one persistent kernel (RZ_VARIANT_MEGA_SINGLE), or (QUEUE) every
//                             segment after the sorted stages when no host-built BVH is there for the tail
// The host (rz_context.cu) runs them in passes sized by the HBM queues between them; by default the tail of the paths —
// what survives the sorted stages — goes to the BVH kernel of rz_bvh_trace.cu instead of K1b.  All use the same
// arithmetic per sphere (rz_sphere_test, packed two spheres per instruction in K1b and two rays per instruction in K1a /
// K1c: rz_search.cuh), the same shading and RNG keys: the image does not depend on the staging.
//
// Execution model of rz_path_kernel
//   * persistent CTAs, grid = SMs x resident CTAs; each WARP pulls work units
//     (32-pixel tile x `chunk` samples, or 512 queue entries) from one global atomic counter;
//   * every lane carries R independent paths ("streams").  When a path ends its stream is
//     REGENERATED at once with the next path of the warp's unit (ballot + popc rank), so the
//     warp-uniform closest-hit loop always runs with full lanes: there is no tail of long
//     paths holding 31 idle lanes;
//   * radiance is accumulated with 64-bit fixed-point (2^-32) integer atomics, so the sum is
//     exact and independent of execution order => bit-identical images for any scheduling,
//     staging and multi-GPU row sharding;
//   * the whole sphere set is staged once per CTA into shared memory with a 1-D bulk
//     async copy (cp.async.bulk + mbarrier, SASS UBLKCP) and searched by brute force with
//     warp-uniform (broadcast) LDS.128 operands and Blackwell packed FP32x2 arithmetic
//     (FFMA2/FADD2/FMUL2, two spheres per instruction): 12 issue slots per stationary
//     sphere PAIR and ray, 15 per moving pair (rz_search_brute2);
//   * large scenes use the BVH kernels of rz_bvh_trace.cu (K3) instead.
#include <algorithm>

#include "rz_launch.h"
#include "rz_search.cuh"

// Resident CTAs per SM the staged kernels are compiled for (register cap = 65536 / (128 * N)); undefined = ptxas decides.
#ifndef RZ_SECOND_MINB
#define RZ_SECOND_MINB 6   // 85 registers.  Round 1 ran 7 CTAs at 72; with the single-copy shading loop that cap costs ~140 B of spills per
#endif                     // thread in the hot loop, and 6 CTAs without spills measured 4.5 % faster (55.1 -> 52.6 ms, scripts/exp_probe.py)
#define RZ_SECOND_BOUNDS __launch_bounds__(128, RZ_SECOND_MINB)
#ifndef RZ_PRIMARY_MINB
#define RZ_PRIMARY_MINB 6   // 85 registers: unconstrained the kernel takes 115 and 4 CTAs (18.2 ms); 5 -> 17.3, 6 -> 16.75, 7 -> 17.0 ms at config 2
#endif
#define RZ_PRIMARY_BOUNDS __launch_bounds__(128, RZ_PRIMARY_MINB)

// per-warp scratch of the sorted-stage kernel: tab[16] u32 | one row of the per-group sphere lists | entry order u32[ue]
__host__ __device__ inline uint32_t rz_second_warp_bytes(uint32_t n_pad, uint32_t ue) {
    return (16u * 4u + rz_bin_row_bytes(n_pad) + 4u * ue + 15u) & ~15u;
}

// ------------------------------------------------------------------------------ the kernel
struct RzStream {
    RzRay ray;
    float3 thr;       // product of attenuations so far (bounceRay's vmul on unwind, renderer.zig:118)
    uint32_t lp;      // local (compact) pixel index -> accumulator slot
    uint32_t gpix;    // global pixel index j*W+i    -> RNG counter
    uint32_t sample;  // global sample index         -> RNG counter
    uint32_t seg;     // segments traced so far (max_bounces - depth of bounceRay)
    bool alive;
};

// G = sphere PAIRS per search-loop iteration
// LIST (not with QUEUE): the adaptive rounds' form, paths of the pixels a.px_list names (RzPathArgs::px_list)
template <int R, int G, bool STATS, int MB, bool QUEUE, bool LIST = false, int SOBOL = 0, bool PASSES = false, bool FILTER = false>
__global__ void __launch_bounds__(128, MB) rz_path_kernel(const RzPathArgs a) {
    extern __shared__ __align__(16) unsigned char rz_smem[];
    __shared__ __align__(8) uint64_t s_bar;
    float4 *s_pk = reinterpret_cast<float4 *>(rz_smem);

    rz_stage_scene_pk(a.set, s_pk, &s_bar);

    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;

    // warp-uniform unit state
    bool have_unit = true;
    uint32_t unit_lp0 = 0, unit_s0 = 0, unit_paths = 0, k_next = 0;
    // QUEUE: paths start from the entries the primary kernel appended (512 per work unit)
    const uint32_t n_entries = QUEUE ? min(*a.q_in_count, a.queue_cap) : 0u;
    const uint32_t n_units = QUEUE ? (n_entries + 511u) / 512u : a.n_units;

    RzStream st[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
        st[r].alive = false;
        st[r].ray.o = f3(0.f, 0.f, 0.f);
        st[r].ray.d = f3(0.f, 1.f, 0.f);
        st[r].ray.time = 0.f;
        st[r].ray.self_k = -1;
        st[r].thr = f3(0.f, 0.f, 0.f);
        st[r].lp = 0; st[r].gpix = 0; st[r].sample = 0; st[r].seg = 0;
    }

    unsigned long long c_paths = 0, c_segs = 0, c_nodes = 0, c_sph = 0, c_hit[3] = {0, 0, 0}, c_sky = 0, c_abs = 0, c_depth = 0;

    while (true) {
        // ---------------------------------------------------------------- regenerate
#pragma unroll
        for (int r = 0; r < R; r++) {
            bool need = !st[r].alive;
            while (true) {
                const unsigned mask = __ballot_sync(0xffffffffu, need);
                if (mask == 0u || !have_unit) break;
                const uint32_t avail = unit_paths - k_next;
                if (avail == 0u) {
                    unsigned u = 0;
                    if (lane == 0) u = atomicAdd(a.unit_counter, 1u);
                    u = __shfl_sync(0xffffffffu, u, 0);
                    if (u >= n_units) { have_unit = false; break; }
                    if (QUEUE) {
                        unit_lp0 = u * 512u;                       // first queue entry of the unit
                        unit_paths = min(512u, n_entries - unit_lp0);
                    } else {
                        const uint32_t tile = u / a.n_chunks, chunk = u - tile * a.n_chunks;
                        unit_lp0 = tile * 32u;
                        unit_s0 = chunk * a.chunk;
                        unit_paths = 32u * min(a.chunk, a.spp - unit_s0);
                    }
                    k_next = 0;
                    continue;
                }
                const uint32_t rank = __popc(mask & lt_mask);
                if (need && rank < avail) {
                    const uint32_t k = k_next + rank;
                    if (QUEUE) {
                        const float4 *e = a.q_in + (size_t)(unit_lp0 + k) * 4u;
                        const float4 qa = __ldcs(e), qb = __ldcs(e + 1), qc = __ldcs(e + 2), qd = __ldcs(e + 3);
                        st[r].ray.o = f3(qa.x, qa.y, qa.z); st[r].ray.time = qa.w;
                        st[r].ray.d = f3(qb.x, qb.y, qb.z); st[r].ray.self_k = __float_as_int(qb.w);
                        st[r].thr = f3(qc.x, qc.y, qc.z); st[r].seg = __float_as_uint(qc.w);
                        st[r].lp = __float_as_uint(qd.x); st[r].gpix = __float_as_uint(qd.y); st[r].sample = __float_as_uint(qd.z);
                        st[r].alive = true;
                        need = false;
                    } else {
                        uint32_t lp = unit_lp0 + (k & 31u);
                        if (lp < (LIST ? a.n_list : a.n_local_px)) {
                            if (LIST) lp = __ldg(a.px_list + lp);
                            uint32_t pi, pj;
                            rz_local_to_global(lp, a.width, a.shard_index, a.shard_count, a.band_rows, pi, pj);
                            st[r].lp = lp;
                            st[r].gpix = pj * a.width + pi;
                            st[r].sample = a.sample_offset + unit_s0 + (k >> 5);
                            st[r].ray = rz_camera_ray(a.cam, pi, pj, st[r].gpix, st[r].sample, a.seed_lo, a.seed_hi, SOBOL, FILTER ? a.sobol : 0u);
                            st[r].thr = f3(1.f, 1.f, 1.f);
                            st[r].seg = 0;
                            st[r].alive = a.max_depth > 0u;
                            if (STATS) { c_paths++; if (!st[r].alive) c_depth++; }
                            need = !st[r].alive;
                        }
                    }
                }
                k_next += min((uint32_t)__popc(mask), avail);
            }
        }
        bool any_alive = false;
#pragma unroll
        for (int r = 0; r < R; r++) any_alive |= st[r].alive;
        if (!__any_sync(0xffffffffu, any_alive)) break;

        // ---------------------------------------------------------------- closest hit
        float bt[R];
        int bk[R];
        RzRay rays[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            bt[r] = 3.0e38f;
            bk[r] = -1;
            rays[r] = st[r].ray;
        }
        rz_search_brute2<R, G>(s_pk, (int)a.set.n_static_pad, (int)a.set.n_pad, rays, a.t_min, bt, bk);

        // ---------------------------------------------------------------- shade
#pragma unroll
        for (int r = 0; r < R; r++) {
            if (!st[r].alive) continue;
            if (STATS) { c_segs++; c_sph += a.set.n; }   // brute force: every sphere of the set
            uint32_t kind;
            const int res = rz_shade_segment(a, st[r].ray, st[r].thr, st[r].seg, st[r].lp, st[r].gpix, st[r].sample, bk[r], kind, SOBOL, PASSES);
            if (STATS) {
                if (kind < 3u) c_hit[kind]++;
                if (res == RZ_END_SKY) c_sky++;
                if (res == RZ_END_ABSORBED) c_abs++;
                if (res == RZ_END_DEPTH) c_depth++;
            }
            if (res != RZ_CONT) st[r].alive = false;
        }
    }

    if (STATS) {
        unsigned long long v[10] = {c_paths, c_segs, c_sph, c_nodes, c_hit[0], c_hit[1], c_hit[2], c_sky, c_abs, c_depth};
#pragma unroll
        for (int i = 0; i < 10; i++) {
            unsigned long long s = v[i];
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0 && s) atomicAdd(&a.stats->v[i], s);
        }
    }
}

// ------------------------------------------------------------------------------ staged kernels: shared pieces
// Code size matters here: the L1.5 instruction cache of an SM holds 32 KB (2048 instructions), the round-1 kernels were
// 40 KB each and ncu charged 3 stall cycles per issued instruction to `no_instruction`.  So everything outside the search
// loop exists ONCE: the two rays a lane carries are shaded by one copy of the code (a two-trip loop that swaps the rays'
// registers), the per-sphere cull is one loop over single spheres for stationary and moving alike, and the rare branches
// (texture walk, unusual diffuse methods) are kept out of line.
struct RzLaneRay {
    RzRay ray;
    float3 thr;
    uint32_t seg, lp, gpix, smp;
    int bk;
    bool live, cont;
    uint32_t key;    // sort key of the scattered ray (when it continues)
};

__device__ __forceinline__ void rz_swap_lane_rays(RzLaneRay &x, RzLaneRay &y) {
    const RzLaneRay t = x;
    x = y;
    y = t;
}

// float <-> int whose signed order is the float's order (for atomicMin / atomicMax on shared memory)
__device__ __forceinline__ int rz_f2ord(float f) { const int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__device__ __forceinline__ float rz_ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

struct RzSegCounters {
    unsigned long long paths, segs, sph, hit[3], sky, abs_, depth;
};

// Shade the two rays of a lane after the search and append the survivors (with their sort keys) to the next queue.
template <bool STATS, int SOBOL, bool PASSES>
__device__ __forceinline__ void rz_shade_and_push2(const RzPathArgs &a, RzLaneRay (&L)[2], unsigned lane, unsigned lt_mask, RzSegCounters &C) {
#pragma unroll 1
    for (int trip = 0; trip < 2; trip++) {
        RzLaneRay &Q = L[0];
        Q.cont = false;
        if (Q.live) {
            if (STATS) C.segs++;
            uint32_t kind;
            const int res = rz_shade_segment(a, Q.ray, Q.thr, Q.seg, Q.lp, Q.gpix, Q.smp, Q.bk, kind, SOBOL, PASSES);
            if (STATS) {
                if (kind < 3u) C.hit[kind]++;
                if (res == RZ_END_SKY) C.sky++;
                if (res == RZ_END_ABSORBED) C.abs_++;
                if (res == RZ_END_DEPTH) C.depth++;
            }
            Q.cont = res == RZ_CONT;
        }
        if (trip == 0) rz_swap_lane_rays(L[0], L[1]);   // ONE exchange per loop: the slots stay swapped afterwards, and nothing below cares which is which
    }
    // ballot-compacted append: one atomic per warp for both rays
    const unsigned m0 = __ballot_sync(0xffffffffu, L[0].cont), m1 = __ballot_sync(0xffffffffu, L[1].cont);
    const unsigned n0 = (unsigned)__popc(m0), n1 = (unsigned)__popc(m1);
    if (n0 + n1 == 0u) return;
    unsigned base = 0;
    if (lane == 0) base = atomicAdd(a.q_out_count, n0 + n1);
    unsigned e = (unsigned)__popc(m0 & lt_mask);
#pragma unroll 1
    for (int trip = 0; trip < 2; trip++) {
        RzLaneRay &Q = L[0];
        // the sort key is computed HERE, between the reservation and the first use of its result: ~100 instructions that hide
        // the round trip of the atomic
        if (Q.cont && a.q_out_keys) Q.key = rz_sort_key(a, Q.ray);
        if (trip == 0) base = __shfl_sync(0xffffffffu, base, 0);
        e += base;
        if (Q.cont) {
            if (e < a.queue_cap) {
                float4 *q = a.q_out + (size_t)e * 4u;
                __stcs(q + 0, make_float4(Q.ray.o.x, Q.ray.o.y, Q.ray.o.z, Q.ray.time));
                __stcs(q + 1, make_float4(Q.ray.d.x, Q.ray.d.y, Q.ray.d.z, __int_as_float(Q.ray.self_k)));
                __stcs(q + 2, make_float4(Q.thr.x, Q.thr.y, Q.thr.z, __uint_as_float(Q.seg)));
                __stcs(q + 3, make_float4(__uint_as_float(Q.lp), __uint_as_float(Q.gpix), __uint_as_float(Q.smp), 0.f));
                if (a.q_out_keys) a.q_out_keys[e] = (unsigned short)Q.key;
            } else {
                atomicOr(a.err, (unsigned)RZ_DEV_ERR_QUEUE_OVERFLOW);   // never silently: the render fails
            }
        }
        if (trip == 0) L[0] = L[1];   // the first ray is stored: only the second one still matters
        e = n0 + (unsigned)__popc(m1 & lt_mask);
    }
}

template <bool STATS>
__device__ __forceinline__ void rz_flush_counters(const RzPathArgs &a, const RzSegCounters &C, unsigned lane) {
    if (!STATS) return;
    const unsigned long long v[10] = {C.paths, C.segs, C.sph, 0ull, C.hit[0], C.hit[1], C.hit[2], C.sky, C.abs_, C.depth};
#pragma unroll 1
    for (int i = 0; i < 10; i++) {
        unsigned long long sum = v[i];
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0 && sum) atomicAdd(&a.stats->v[i], sum);
    }
}

// ------------------------------------------------------------------------------ primary kernel
// Stage 1 of the staged K1: the camera segment of every path (Camera.getRay camera.zig:59-77 + the first
// bounceRay level renderer.zig:103-126).  Camera rays of a 32-pixel tile are coherent, so the warp first
// culls the sphere set against the tile's frustum — a cone around the tile's mean direction, widened by the
// pixel footprint, the thin-lens blur and each sphere's motion — and the packed search then runs over the
// surviving handful of spheres instead of all of them (rz_search_lists_r2: same arithmetic, same (t, k)).
// Paths that scatter are appended, ballot-compacted, to the HBM queue the sorted stages start from; paths
// that leave the scene or are absorbed accumulate here.  36 % of all segments are camera segments.  The cull
// (rz_tile_cone / rz_tile_keep, rz_device.cuh) is host + device and property-tested on the CPU.
template <bool STATS, int SOBOL = 0, bool PASSES = false, bool FILTER = false>
__global__ void RZ_PRIMARY_BOUNDS rz_primary_kernel(const RzPathArgs a) {
    extern __shared__ __align__(16) unsigned char rz_smem[];
    __shared__ __align__(8) uint64_t s_bar;
    float4 *s_cr = reinterpret_cast<float4 *>(rz_smem);
    const uint32_t cv_f4 = 2u * a.set.n_pad - a.set.n_static_pad;
    unsigned short *ls = reinterpret_cast<unsigned short *>(s_cr + cv_f4) + (threadIdx.x >> 5) * a.set.n_pad;   // kept stationary spheres
    unsigned short *lm = ls + a.set.n_static_pad;                                                               // kept moving spheres

    const float4 *s_vel = rz_stage_scene_cv(a.set, s_cr, &s_bar);

    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    RzSegCounters C = {};

    while (true) {
        unsigned u = 0;
        if (lane == 0) u = atomicAdd(a.unit_counter, 1u);
        u = __shfl_sync(0xffffffffu, u, 0);
        if (u >= a.n_units) break;
        u += a.unit_base;
        const uint32_t tile = u / a.n_chunks, chunk = u - tile * a.n_chunks;
        const uint32_t lp = tile * 32u + lane;
        const bool valid = lp < a.n_local_px;
        uint32_t pi = 0, pj = 0;
        if (valid) rz_local_to_global(lp, a.width, a.shard_index, a.shard_count, a.band_rows, pi, pj);
        const uint32_t gpix = pj * a.width + pi;

        // ---- cone around the tile's camera rays: axis = mean pixel direction, half-angle from the pixel corners (under a pixel
        // filter, the corners of the support its samples reach)
        const float3 pc = rz_tile_pixel_dir(a.cam, pi, pj);
        float3 ax = valid ? normalize3(pc) : f3(0.f, 0.f, 0.f);
        for (int o = 16; o > 0; o >>= 1) {
            ax.x += __shfl_xor_sync(0xffffffffu, ax.x, o); ax.y += __shfl_xor_sync(0xffffffffu, ax.y, o); ax.z += __shfl_xor_sync(0xffffffffu, ax.z, o);
        }
        const bool has_axis = rz_tile_axis(ax);
        float cmin = valid ? rz_tile_corner_cos(a.cam, pc, ax, FILTER ? rz_filter_reach(a.sobol) : 0.5f) : 1.0f;
        for (int o = 16; o > 0; o >>= 1) cmin = fminf(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
        const RzTileCone cone = rz_tile_cone(a.cam, ax, has_axis, cmin, a.focus_dist, a.lens_radius);
        // one lane per sphere, stationary and moving through the same code; the lists keep set order (= search order)
        int n_ls = 0, n_lm = 0;
#pragma unroll 1
        for (uint32_t k0 = 0; k0 < a.set.n_pad; k0 += 32u) {
            const uint32_t k = k0 + lane;
            const bool st = k < a.set.n_static_pad;
            float4 S = make_float4(0.f, 0.f, 0.f, 1.f), V = make_float4(0.f, 0.f, 0.f, 0.f);   // lanes past the set: a padding entry
            if (k < a.set.n_pad) { S = s_cr[k]; if (!st) V = s_vel[k]; }
            const bool keep = k < a.set.n_pad && rz_tile_keep(cone, S.x, S.y, S.z, V.x, V.y, V.z, S.w);
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            const unsigned ms = m & __ballot_sync(0xffffffffu, st);
            if (keep && st) ls[n_ls + __popc(ms & lt_mask)] = (unsigned short)k;
            if (keep && !st) lm[n_lm + __popc((m & ~ms) & lt_mask)] = (unsigned short)k;
            n_ls += __popc(ms); n_lm += __popc(m & ~ms);
        }
        __syncwarp();

        // ---- the tile's samples of this chunk, two per lane and iteration
        const uint32_t s0 = chunk * a.chunk, ns = min(a.chunk, a.spp - s0);
#pragma unroll 1
        for (uint32_t s = 0; s < ns; s += 2u) {
            RzLaneRay L[2];
#pragma unroll 1
            for (int trip = 0; trip < 2; trip++) {                  // one copy of the camera-ray code for both rays
                RzLaneRay &Q = L[0];
                Q.smp = a.sample_offset + s0 + s + (uint32_t)trip;
                const bool have = valid && (s + (uint32_t)trip < ns);
                Q.live = have && a.max_depth > 0u;
                if (STATS && have) { C.paths++; if (!Q.live) C.depth++; }
                if (Q.live) Q.ray = rz_camera_ray(a.cam, pi, pj, gpix, Q.smp, a.seed_lo, a.seed_hi, SOBOL, FILTER ? a.sobol : 0u);
                else { Q.ray.o = f3(0.f, 0.f, 0.f); Q.ray.d = f3(0.f, 1.f, 0.f); Q.ray.time = 0.f; Q.ray.self_k = -1; }
                Q.thr = f3(1.f, 1.f, 1.f); Q.seg = 0u; Q.lp = lp; Q.gpix = gpix; Q.bk = -1; Q.cont = false; Q.key = 0u;
                if (trip == 0) L[1] = L[0];   // slot 0 is rewritten by the second trip
            }
            {
                RzRay rays[2] = {L[0].ray, L[1].ray};
                float bt[2] = {3.0e38f, 3.0e38f};
                int bk[2] = {-1, -1};
                rz_search_lists_r2(s_cr, s_vel, ls, n_ls, lm, n_lm, rays, a.t_min, bt, bk);
                L[0].ray = rays[0]; L[1].ray = rays[1];   // (the search holds o, d, time as packed pairs and hands them back)
                L[0].bk = bk[0]; L[1].bk = bk[1];
            }
            if (STATS) C.sph += (unsigned long long)(n_ls + n_lm) * ((L[0].live ? 1u : 0u) + (L[1].live ? 1u : 0u));
            rz_shade_and_push2<STATS, SOBOL, PASSES>(a, L, lane, lt_mask, C);
        }
        __syncwarp();   // the lists are rewritten for the next unit
    }
    rz_flush_counters<STATS>(a, C, lane);
}

// ------------------------------------------------------------------------------ per-group sphere lists
// For every group of the sort — (origin cell, direction field) = the top 12 bits of rz_sort_key — the spheres a ray of that
// group can reach, ordered by the SMALLEST reach class that gets to them (rz_unit_class: class 16 = no ray of the group
// can, the sphere is left out; inside a class, set order).  Camera-independent: a function of the sphere set and the key grid
// only; one warp per group, ~30 us for the 4096 groups, run at the start of every staged render.  The sorted-segment kernel
// copies a row per work unit instead of classifying the set itself (round 2's first form did: ~15 % of its samples, and it
// had to merge the bounds of every key in the unit, which is looser than one group's own).  Row layout: rz_bin_row_bytes.
__global__ void __launch_bounds__(128) rz_bin_lists_kernel(const RzPathArgs a) {
    extern __shared__ __align__(16) unsigned char rz_smem[];
    __shared__ __align__(8) uint64_t s_bar;
    float4 *s_cr = reinterpret_cast<float4 *>(rz_smem);
    const uint32_t cv_f4 = 2u * a.set.n_pad - a.set.n_static_pad;
    // per-warp scratch: tab[32] (spheres per class: stationary, moving) | sphere classes u8[n_pad]
    const uint32_t warp_bytes = (32u * 4u + a.set.n_pad + 15u) & ~15u;
    unsigned char *wb = reinterpret_cast<unsigned char *>(s_cr + cv_f4) + (threadIdx.x >> 5) * warp_bytes;
    unsigned int *tab = reinterpret_cast<unsigned int *>(wb);
    unsigned char *scl = wb + 32u * 4u;
    const float4 *s_vel = rz_stage_scene_cv(a.set, s_cr, &s_bar);
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    for (uint32_t bin = blockIdx.x * 4u + (threadIdx.x >> 5); bin < (uint32_t)RZ_SORT_BINS; bin += gridDim.x * 4u) {
        RzUnitBounds U;
        rz_unit_bounds_init(U);
        rz_unit_bounds_add_cell(U, a, bin << 4);
        unsigned short *row = reinterpret_cast<unsigned short *>(a.bin_lists + (size_t)bin * a.bin_row);
        unsigned short *ls = row + 32, *lm = ls + a.set.n_static_pad;
        tab[lane] = 0u;
        __syncwarp();
        // smallest class that reaches each sphere (one lane per sphere)
#pragma unroll 1
        for (uint32_t k0 = 0; k0 < a.set.n_pad; k0 += 32u) {
            const uint32_t k = k0 + lane;
            if (k < a.set.n_pad) {
                const bool st = k < a.set.n_static_pad;
                const float4 S = s_cr[k];
                float4 V = make_float4(0.f, 0.f, 0.f, 0.f);
                if (!st) V = s_vel[k];
                const int c = rz_unit_class(U, a, S.x, S.y, S.z, V.x, V.y, V.z, S.w);
                scl[k] = (unsigned char)c;
                if (c < 16) atomicAdd(&tab[(st ? 0u : 16u) + (uint32_t)c], 1u);
            }
        }
        __syncwarp();
        {   // inclusive prefixes of the two histograms -> the row's end_s / end_m; exclusive ones -> running cursors
            const uint32_t cnt = tab[lane];                                  // lanes 0-15: stationary, 16-31: moving
            uint32_t inc = cnt;
            for (int o = 1; o < 16; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if ((int)(lane & 15u) >= o) inc += t; }
            __syncwarp();
            tab[lane] = inc - cnt;
            row[lane] = (unsigned short)inc;
        }
        __syncwarp();
#pragma unroll 1
        for (uint32_t k0 = 0; k0 < a.set.n_pad; k0 += 32u) {
            const uint32_t k = k0 + lane;
            const bool st = k < a.set.n_static_pad;
            const uint32_t c = k < a.set.n_pad ? (uint32_t)scl[k] : 16u;
            const uint32_t tag = c < 16u ? (c | (st ? 0u : 16u)) : 32u + lane;   // (part, class); unique for spheres that are dropped
            const unsigned peers = __match_any_sync(0xffffffffu, tag);
            const int leader = __ffs((int)peers) - 1;
            uint32_t base = 0u;
            if ((int)lane == leader && c < 16u) { base = tab[tag]; tab[tag] = base + (uint32_t)__popc(peers); }
            base = __shfl_sync(0xffffffffu, base, leader);
            if (c < 16u) (st ? ls : lm)[base + (uint32_t)__popc(peers & lt_mask)] = (unsigned short)k;
            __syncwarp();
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------ sorted-segment kernel
// The stages after the camera segment, one launch per segment (segments 2..6 by default).  Scattered rays are incoherent,
// but their queue entries have been GROUPED by (origin cell, direction field) — the top 12 bits of rz_sort_key, rz_sort.cu —
// and the sort has cut every group into work units of at most `ue` entries, so the rays of a unit start in one cell and head
// the same way.  Per unit the warp
//   1. finds the unit's group (three warp-wide probes of the sort's unit prefix) and copies the group's row of pair lists
//      (rz_bin_lists_kernel): the sphere pairs its rays can reach, ordered by the smallest reach class that gets to them;
//   2. orders the unit's entries by the key's low 4 bits, the reach class — how long a ray stays inside the box around the
//      non-huge spheres (a counting sort over 16 classes in shared memory);
//   3. takes the entries 64 at a time in class order: a batch whose largest class is c searches the pairs of classes <= c, a
//      prefix of the ordered pair list (rz_search_list2: the same arithmetic per sphere, so (t, k) is unchanged).
// Round 1 sorted on all 16 key bits (two radix passes) and culled each unit with its largest reach; ordering by reach
// inside the unit costs one global pass less and culls every batch with its OWN reach.  The cull functions are host +
// device and property-tested on the CPU (tests/test_hostsim_cpu.py).
template <bool STATS, int SOBOL = 0, bool PASSES = false>
__global__ void RZ_SECOND_BOUNDS rz_second_kernel(const RzPathArgs a) {
    extern __shared__ __align__(16) unsigned char rz_smem[];
    __shared__ __align__(8) uint64_t s_bar;
    float4 *s_cr = reinterpret_cast<float4 *>(rz_smem);
    const uint32_t cv_f4 = 2u * a.set.n_pad - a.set.n_static_pad;
    const uint32_t ue_max = a.unit_entries;
    // per-warp scratch: tab[16] | the group's row (end_s, end_m, ls, lm) | entry order [ue] (layout: rz_second_warp_bytes)
    const uint32_t warp_bytes = rz_second_warp_bytes(a.set.n_pad, ue_max);
    unsigned char *wb = reinterpret_cast<unsigned char *>(s_cr + cv_f4) + (threadIdx.x >> 5) * warp_bytes;
    unsigned int *tab = reinterpret_cast<unsigned int *>(wb);             // [0,16) entries: end of class c
    unsigned short *row = reinterpret_cast<unsigned short *>(tab + 16);   // end_s[16] end_m[16]: spheres of classes <= c
    unsigned short *ls = row + 32;
    unsigned short *lm = ls + a.set.n_static_pad;
    uint32_t *order = reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(row) + a.bin_row);   // queue entry indices in class order

    const float4 *s_vel = rz_stage_scene_cv(a.set, s_cr, &s_bar);

    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned int *bin_end = a.q_in_bins, *unit_first = a.q_in_bins + RZ_BIN_UNIT_FIRST;
    const uint32_t n_units = unit_first[RZ_SORT_BINS], ue = min(a.q_in_bins[RZ_BIN_UE], ue_max);
    RzSegCounters C = {};

    while (true) {
        unsigned u = 0;
        if (lane == 0) u = atomicAdd(a.unit_counter, 1u);
        u = __shfl_sync(0xffffffffu, u, 0);
        if (u >= n_units) break;
        // ---- 1. the unit's group: the last b with unit_first[b] <= u (groups without entries share their successor's value)
        uint32_t bin = 0u;
#pragma unroll
        for (uint32_t stride = 128u; stride; stride = stride == 128u ? 4u : stride == 4u ? 1u : 0u) {
            const uint32_t i = bin + lane * stride;
            const bool le = (stride > 1u || lane < 4u) && unit_first[i] <= u;       // unit_first[bin] <= u always: lane 0 votes yes
            bin += ((uint32_t)__popc(__ballot_sync(0xffffffffu, le)) - 1u) * stride;
        }
        const uint32_t g0 = bin ? bin_end[bin - 1u] : 0u;                          // after the scatter: bins[b] = end of group b
        const uint32_t e0 = g0 + (u - unit_first[bin]) * ue, ne = min(ue, bin_end[bin] - e0);
        const uint32_t *uidx = a.q_in_idx + e0;   // entry index | class << 28
        {   // the group's row -> shared memory (16-byte pieces; the table stays in L2)
            const uint4 *src = reinterpret_cast<const uint4 *>(a.bin_lists + (size_t)bin * a.bin_row);
            uint4 *dst = reinterpret_cast<uint4 *>(row);
            for (uint32_t i = lane; i < a.bin_row / 16u; i += 32u) dst[i] = __ldg(src + i);
        }
        // ---- 2. rays per reach class, then the entries in class order
        if (lane < 16u) tab[lane] = 0u;
        __syncwarp();
#pragma unroll 1
        for (uint32_t i0 = 0; i0 < ne; i0 += 128u) {   // four keys in flight per lane: the loop is pure load latency otherwise
            uint32_t kc[4];
#pragma unroll
            for (int j = 0; j < 4; j++) { const uint32_t i = i0 + 32u * (uint32_t)j + lane; kc[j] = i < ne ? (uidx[i] >> RZ_IDX_CLASS_SHIFT) : 16u; }
#pragma unroll
            for (int j = 0; j < 4; j++) if (kc[j] < 16u) atomicAdd(&tab[kc[j]], 1u);
        }
        __syncwarp();
        {   // exclusive prefix over the 16 classes -> running cursors
            const uint32_t cnt = lane < 16u ? tab[lane] : 0u;
            uint32_t inc = cnt;
            for (int o = 1; o < 16; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if ((int)lane >= o) inc += t; }
            __syncwarp();
            if (lane < 16u) tab[lane] = inc - cnt;
        }
        __syncwarp();
        // order[slot] = queue entry (read here, coalesced, so that the batches below go from shared memory straight to the
        // entry).  Lanes with the same class take consecutive slots.
#pragma unroll 1
        for (uint32_t i0 = 0; i0 < ne; i0 += 128u) {
            uint32_t ke[4];
#pragma unroll
            for (int j = 0; j < 4; j++) { const uint32_t i = i0 + 32u * (uint32_t)j + lane; ke[j] = i < ne ? uidx[i] : 0xffffffffu; }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t c = ke[j] != 0xffffffffu ? (ke[j] >> RZ_IDX_CLASS_SHIFT) : 16u + lane;
                const unsigned peers = __match_any_sync(0xffffffffu, c);
                const int leader = __ffs((int)peers) - 1;
                uint32_t base = 0u;
                if ((int)lane == leader && c < 16u) { base = tab[c]; tab[c] = base + (uint32_t)__popc(peers); }
                base = __shfl_sync(0xffffffffu, base, leader);
                if (c < 16u) order[base + (uint32_t)__popc(peers & lt_mask)] = ke[j] & RZ_IDX_MASK;
                __syncwarp();
            }
        }
        // now tab[c] = end of class c in `order`

        // ---- 3. the unit's rays in class order, two per lane and iteration
#pragma unroll 1
        for (uint32_t b0 = 0; b0 < ne; b0 += 64u) {
            // the batch's largest class: that of its last entry = number of classes that end at or before it
            const uint32_t last = min(b0 + 63u, ne - 1u);
            const int cmax = min(15, __popc(__ballot_sync(0xffffffffu, lane < 16u && tab[lane] <= last)));
            const int n_ls = (int)row[cmax], n_lm = (int)row[16 + cmax];
            RzLaneRay L[2];
            {   // both rays' entries are fetched together: eight 16-byte loads in flight per lane (random 64 B gathers from HBM)
                const float4 *e[2];
                float4 qa[2], qb[2], qc[2], qd[2];
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    const uint32_t j = b0 + lane + 32u * (uint32_t)r;
                    L[r].live = j < ne;
                    e[r] = a.q_in + (size_t)(L[r].live ? order[j] : 0u) * 4u;
                }
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    if (L[r].live) { qa[r] = __ldcs(e[r]); qb[r] = __ldcs(e[r] + 1); qc[r] = __ldcs(e[r] + 2); qd[r] = __ldcs(e[r] + 3); }
                    else { qa[r] = make_float4(0.f, 0.f, 0.f, 0.f); qb[r] = make_float4(0.f, 1.f, 0.f, __int_as_float(-1)); qc[r] = qa[r]; qd[r] = qa[r]; }
                }
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    RzLaneRay &Q = L[r];
                    Q.ray.o = f3(qa[r].x, qa[r].y, qa[r].z); Q.ray.time = qa[r].w;
                    Q.ray.d = f3(qb[r].x, qb[r].y, qb[r].z); Q.ray.self_k = __float_as_int(qb[r].w);
                    Q.thr = f3(qc[r].x, qc[r].y, qc[r].z); Q.seg = __float_as_uint(qc[r].w);
                    Q.lp = __float_as_uint(qd[r].x); Q.gpix = __float_as_uint(qd[r].y); Q.smp = __float_as_uint(qd[r].z);
                    Q.bk = -1; Q.cont = false; Q.key = 0u;
                }
            }
            {
                RzRay rays[2] = {L[0].ray, L[1].ray};
                float bt[2] = {3.0e38f, 3.0e38f};
                int bk[2] = {-1, -1};
                rz_search_lists_r2(s_cr, s_vel, ls, n_ls, lm, n_lm, rays, a.t_min, bt, bk);
                L[0].ray = rays[0]; L[1].ray = rays[1];   // (the search holds o, d, time as packed pairs and hands them back)
                L[0].bk = bk[0]; L[1].bk = bk[1];
            }
            if (STATS) C.sph += (unsigned long long)(n_ls + n_lm) * ((L[0].live ? 1u : 0u) + (L[1].live ? 1u : 0u));
            rz_shade_and_push2<STATS, SOBOL, PASSES>(a, L, lane, lt_mask, C);
        }
        __syncwarp();
    }
    rz_flush_counters<STATS>(a, C, lane);
}

// ------------------------------------------------------------------------------ launchers
static size_t rz_pk_bytes(const RzPathArgs &a) { return (size_t)(a.set.n_pad + (a.set.n_pad - a.set.n_static_pad)) * 16u; }

// Shared memory the sorted-stage kernel needs: the set + per-warp scratch (rz_second_warp_bytes).
static size_t rz_second_smem_bytes(const RzPathArgs &a) {
    return rz_pk_bytes(a) + 4u * (size_t)rz_second_warp_bytes(a.set.n_pad, a.unit_entries);
}

static auto rz_second_instance(const RzPathArgs &a, int collect_stats) {
    return rz_pick_instance(a, collect_stats, [](auto S, auto M, auto P) { return rz_second_kernel<decltype(S)::value, decltype(M)::value, decltype(P)::value>; });
}

// One form of rz_path_kernel on the persistent grid; rays_per_thread in {1,2}.
template <bool QUEUE, bool LIST>
static cudaError_t rz_launch_one(const RzPathArgs &a, int rays_per_thread, int collect_stats, int sm_count, cudaStream_t stream,
                                 int *grid_out) {
    // the forms that generate camera rays have FILTER instances (rz_pick_camera_instance); the queue-fed form does not
    auto pick = [&](auto inst) {
        if constexpr (QUEUE) return rz_pick_instance(a, collect_stats, [inst](auto S, auto M, auto P) { return inst(S, M, P, std::false_type{}); });
        else return rz_pick_camera_instance(a, collect_stats, inst);
    };
    const auto one = pick([](auto S, auto M, auto P, auto F) {
        return rz_path_kernel<1, 2, decltype(S)::value, 5, QUEUE, LIST, decltype(M)::value, decltype(P)::value, decltype(F)::value>;
    });
    // 8 resident CTAs per SM (64 registers, 232 B of spills outside the search loop) measured 3 % faster than the 5 CTAs the
    // unconstrained 88-register build gets: 1522 vs 1472 Mpaths/s at config 2 / 100 spp.  (The STATS instances keep 5.)
    const auto two = pick([](auto S, auto M, auto P, auto F) {
        return rz_path_kernel<2, 2, decltype(S)::value, decltype(S)::value ? 5 : 8, QUEUE, LIST, decltype(M)::value, decltype(P)::value, decltype(F)::value>;
    });
    const auto kern = rays_per_thread == 1 ? one : two;
    const size_t smem = rz_pk_bytes(a);
    int grid = 0;
    const cudaError_t e = rz_persistent_grid(kern, smem, sm_count, &grid);
    if (e != cudaSuccess) return e;
    if (grid_out) *grid_out = grid;
    kern<<<grid, 128, smem, stream>>>(a);
    return cudaGetLastError();
}

// Forces the lazily loaded path kernels into the context (called once from rayz_cuda_create so that
// the first render does not pay module loading).
extern "C" cudaError_t rz_path_warm(void) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, rz_path_kernel<2, 2, false, 8, true>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, rz_primary_kernel<false>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, rz_second_kernel<false>);
    return e;
}

// Shared memory the primary kernel needs: the pair-interleaved set + one pair list per warp.
extern "C" size_t rz_primary_smem_bytes(const RzPathArgs *a) {
    return rz_pk_bytes(*a) + ((4u * (size_t)a->set.n_pad * sizeof(unsigned short) + 15u) & ~size_t(15));
}

// Stage 1: camera segments of the work units [unit_base, unit_base + n_units) -> queue.
extern "C" cudaError_t rz_launch_primary(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream) {
    const auto kern = rz_pick_camera_instance(*a, collect_stats, [](auto S, auto M, auto P, auto F) {
        return rz_primary_kernel<decltype(S)::value, decltype(M)::value, decltype(P)::value, decltype(F)::value>;
    });
    const size_t smem = rz_primary_smem_bytes(a);
    int grid = 0;
    const cudaError_t e = rz_persistent_grid(kern, smem, sm_count, &grid);
    if (e != cudaSuccess) return e;
    const unsigned want = (a->n_units + 3u) / 4u;   // 4 warps per CTA, one unit per warp at a time
    kern<<<std::max(1u, std::min((unsigned)grid, want)), 128, smem, stream>>>(*a);
    return cudaGetLastError();
}

// Per-group pair lists of the sorted-segment kernel (a->bin_lists: RZ_SORT_BINS rows of a->bin_row bytes).
extern "C" cudaError_t rz_launch_bin_lists(const RzPathArgs *a, int sm_count, cudaStream_t stream) {
    const size_t smem = rz_pk_bytes(*a) + 4u * (size_t)((32u * 4u + a->set.n_pad + 15u) & ~15u);
    cudaError_t e = cudaFuncSetAttribute(rz_bin_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    rz_bin_lists_kernel<<<std::min(RZ_SORT_BINS / 4, sm_count * 4), 128, smem, stream>>>(*a);
    return cudaGetLastError();
}

// Grid size of the sorted-segment kernel (the sort sizes the work units with it).
extern "C" cudaError_t rz_second_grid(const RzPathArgs *a, int collect_stats, int sm_count, int *grid) {
    return rz_persistent_grid(rz_second_instance(*a, collect_stats), rz_second_smem_bytes(*a), sm_count, grid);
}

// Stage 2: second segments of the sorted queue (q_in through q_in_idx) -> q_out.
extern "C" cudaError_t rz_launch_second(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream) {
    int grid = 0;
    const cudaError_t e = rz_second_grid(a, collect_stats, sm_count, &grid);
    if (e != cudaSuccess) return e;
    rz_second_instance(*a, collect_stats)<<<grid, 128, rz_second_smem_bytes(*a), stream>>>(*a);
    return cudaGetLastError();
}

// Last stage (q_in != nullptr): the persistent megakernel started from a queue; or the single-stage form
// (q_in == nullptr) that generates its own camera rays (of the pixels of px_list when it is set).  rays_per_thread in {1,2}.
extern "C" cudaError_t rz_launch_path(const RzPathArgs *a, int rays_per_thread, int collect_stats, int sm_count, cudaStream_t stream,
                                      int *grid_out) {
    if (a->q_in) return rz_launch_one<true, false>(*a, rays_per_thread, collect_stats, sm_count, stream, grid_out);
    if (a->px_list)   // an adaptive round: the same instances over the listed pixels
        return rz_launch_one<false, true>(*a, rays_per_thread, collect_stats, sm_count, stream, grid_out);
    return rz_launch_one<false, false>(*a, rays_per_thread, collect_stats, sm_count, stream, grid_out);
}
