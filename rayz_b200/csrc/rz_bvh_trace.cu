// rz_bvh_trace.cu — K3: persistent BVH path kernel for scenes that do not fit the brute-force kernel
// (and the fastest variant in paths/s on small ones).
//
// Restates the role of BVH.findHit + AABB.hit (reference src/hit.zig:70-98, 181-216) inside the path
// loop of renderer.zig:85-126.  The reference recurses per ray, left child first; here every lane of
// a persistent warp walks its own ray through a flattened BVH2 (both child boxes in the parent, 64 B,
// read through ld.global.nc), near child first, with an explicit per-lane stack.  (A 4-wide tree was measured and
// rejected: DESIGN.md section 3, "K3 and the wide BVH".)
//
// What shapes the kernel is SIMT divergence, not arithmetic: the first version (per-lane
// `while (stack)` with the leaf tests nested inside, rays replaced only between segments) ran with
// 7.4-9.4 of 32 lanes active per instruction at 80 % issue utilisation (ncu, profiles/).  Hence:
//   * while-while traversal (Aila & Laine, HPG 2009): an inner loop that only descends through
//     internal nodes, then a leaf phase that all lanes holding a leaf execute together;
//   * ray replacement INSIDE the traversal loop: as soon as fewer than ACTIVE_MIN lanes are still
//     traversing, the finished lanes shade their hit, scatter or start the next (pixel, sample) of
//     the warp's work unit, and rejoin — instead of idling until the slowest ray of the warp ends;
//   * a descend round ends as soon as fewer than DESCEND_MIN lanes are still descending, so lanes that
//     hold a leaf do not idle behind a few long descents (the interrupted lanes resume next round);
//   * leaves are pushed on the stack like nodes (encoded negative), so a popped leaf is handled by the
//     same leaf phase.
// Measured on B200 (config-2 scene / 99,856 spheres, Mpaths/s): first version 2245 / 903; while-while +
// replacement at ACTIVE_MIN = 8: 2640 / 1241; + DESCEND_MIN = 24: 3370 / 1547; + one sphere per LBVH leaf
// (rz_bvh_build.cu) and the two children's slab arithmetic packed into FP32x2 (6 FADD2 + 6 FMUL2 per node
// visit instead of 24 scalar instructions, bit-identical per half): 3774 / 1931; + child references finalized
// at upload (rz_bvh_finalize: nothing to decode or check per visit): 3974 / 2025; + 8 resident CTAs (RZ_BVH_MINB: the walk waits
// on node loads from L2, warps pay more than registers): 4249 / 2139; + tile lists in the camera stage (rz_bvh_stage_kernel:
// the tree culled once per 8 x 4-pixel block against the block's cone, the block's rays search the surviving spheres as a list):
// 4813 / 2497.  Picking the near/far planes by ray-direction sign (six 8-byte loads instead of three 16-byte loads and twelve
// min/max) was 9 % SLOWER and is not used; so were a branch-free node visit, a deferred leaf phase, a pending-leaf slot and an
// L1 prefetch of the deferred child (profiles/r02_experiments.md expb7-expb10).
// Sphere tests, hit refinement, shading, RNG keys and accumulation are the shared device functions of
// rz_search.cuh / rz_device.cuh: two trees give bit-identical images; against a brute-force search a pixel or two may
// differ (the FP32 sphere test has a fuzzy surface, the boxes are exact: a grazing ray can "hit" a sphere a hair outside
// its box, which brute force tests and the tree prunes — tests/test_gpu_parity.py bounds it at <= 3 pixels).
#include "rz_launch.h"
#include "rz_search.cuh"

namespace {

constexpr int RZ_SENTINEL = 0x7fffffff;
// Resident CTAs per SM the BVH kernels are compiled for (register cap 65536 / (128 * N)).  On the 99,856-sphere scene the traversal
// waits on node loads from L2 (ncu, profiles/r02_bvh_kernel_config4_ncu.md: 2.9 long-scoreboard stall cycles per issued
// instruction at 24 resident warps, 16 % of the samples on the first use of a node), so warps pay more than registers: 8 CTAs at
// 64 registers (56 B of spills) beat 6 CTAs at 78 without spills.  Config 4 / BVH variant on config 2, Mpaths/s: 5 or 6 CTAs
// 2027 / 3974, 7 -> 2126 / 4198, 8 -> 2139 / 4249, 9 -> 2115 / 4206, 10 -> 1880 / 3667 (profiles/r02_experiments.md expb6).
#ifndef RZ_BVH_MINB
#define RZ_BVH_MINB 8
#endif
#ifndef RZ_BVH_CAMERA_MINB
#define RZ_BVH_CAMERA_MINB 6   // resident CTAs of the camera stage with tile lists: cull + packed search + shading + the per-ray walk in one kernel
#endif
#ifndef RZ_CL_CAP
#define RZ_CL_CAP 256          // spheres a tile's list can hold (more: the tile's rays walk the tree)
#endif
#ifndef RZ_CL_WL
#define RZ_CL_WL 256           // nodes in flight during the cull (ring buffer; power of two)
#endif
constexpr int RZ_STACK = 96;   // LBVH depth bound: 63 Morton bits + 32 index tie-break bits

// One while-while round for this lane's ray: descend through internal nodes to the next leaf (or until the warp's round
// is cut short), then test that leaf.  Shared by the persistent kernel and the staged (sorted) kernels.
template <bool STATS>
__device__ __forceinline__ void rz_bvh_round(const RzPathArgs &a, const float4 *__restrict__ nodes, const RzRay &ray, float ix, float iy,
                                             float iz, int &cur, int &sp, int (&stack)[RZ_STACK], float &bt, int &bk, int descend_min,
                                             unsigned long long &c_nodes, unsigned long long &c_sph) {
    // (1) descend through internal nodes until this lane holds a leaf or runs dry; the round ends early
    //     once fewer than `descend_min` lanes are still descending, so that lanes holding a leaf do not idle
    //     behind a few long descents (those lanes simply resume in the next round)
    while ((unsigned)cur < (unsigned)RZ_SENTINEL) {
        // slab test of AABB.hit (hit.zig:70-98) with multiply-by-inverse; boxes are padded outward at build time
        float tn0, tf0, tn1, tf1;
        int4 q3;
        if (STATS) c_nodes += 2;
        const float ox = ray.o.x, oy = ray.o.y, oz = ray.o.z;
        {
            const float4 q0 = __ldg(nodes + cur * 4 + 0);  // lox0 lox1 hix0 hix1
            const float4 q1 = __ldg(nodes + cur * 4 + 1);  // loy0 loy1 hiy0 hiy1
            const float4 q2 = __ldg(nodes + cur * 4 + 2);  // loz0 loz1 hiz0 hiz1
            q3 = __ldg(reinterpret_cast<const int4 *>(nodes + cur * 4 + 3));
            // the two children's planes sit side by side in the node, so (plane - o) * inv_d is one FADD2 + one FMUL2 for both
            // (packed FP32x2, the ray's operands as broadcasts): 12 issue slots instead of 24, the same IEEE operations per half
            float ax0, ax1, bx0, bx1, ay0, ay1, by0, by1, az0, az1, bz0, bz1;
            const rz_p2 nox = rz_pack(-ox, -ox), noy = rz_pack(-oy, -oy), noz = rz_pack(-oz, -oz);
            const rz_p2 ix2 = rz_pack(ix, ix), iy2 = rz_pack(iy, iy), iz2 = rz_pack(iz, iz);
            rz_unpack(rz_mul2(rz_add2(rz_pack(q0.x, q0.y), nox), ix2), ax0, ax1);
            rz_unpack(rz_mul2(rz_add2(rz_pack(q0.z, q0.w), nox), ix2), bx0, bx1);
            rz_unpack(rz_mul2(rz_add2(rz_pack(q1.x, q1.y), noy), iy2), ay0, ay1);
            rz_unpack(rz_mul2(rz_add2(rz_pack(q1.z, q1.w), noy), iy2), by0, by1);
            rz_unpack(rz_mul2(rz_add2(rz_pack(q2.x, q2.y), noz), iz2), az0, az1);
            rz_unpack(rz_mul2(rz_add2(rz_pack(q2.z, q2.w), noz), iz2), bz0, bz1);
            tn0 = fmaxf(fmaxf(fminf(ax0, bx0), fminf(ay0, by0)), fmaxf(fminf(az0, bz0), a.t_min));
            tf0 = fminf(fminf(fmaxf(ax0, bx0), fmaxf(ay0, by0)), fminf(fmaxf(az0, bz0), bt));
            tn1 = fmaxf(fmaxf(fminf(ax1, bx1), fminf(ay1, by1)), fmaxf(fminf(az1, bz1), a.t_min));
            tf1 = fminf(fminf(fmaxf(ax1, bx1), fmaxf(ay1, by1)), fminf(fmaxf(az1, bz1), bt));
        }
        const bool h0 = tn0 <= tf0 * 1.0000004f, h1 = tn1 <= tf1 * 1.0000004f;
        // child references as rz_bvh_finalize left them in the node: internal index >= 0, or a leaf (rz_leaf_ref: negative, carries
        // its count); there are no unused slots (round 2's first form decoded (child, count) here: 12 of ~63 instructions per visit)
        const int c0 = q3.x, c1 = q3.y;
        if (h0 && h1) {
            const bool swap = tn1 < tn0;
            if (sp < (int)a.stack_cap) stack[sp++] = swap ? c0 : c1;
            else atomicOr(a.err, (unsigned)RZ_DEV_ERR_STACK_OVERFLOW);   // a dropped subtree would darken the image silently
            cur = swap ? c1 : c0;
        } else if (h0) {
            cur = c0;
        } else if (h1) {
            cur = c1;
        } else {
            cur = sp > 0 ? stack[--sp] : RZ_SENTINEL;
        }
        if (__popc(__activemask()) < descend_min) break;
    }
    // (2) leaf phase
    if (cur < 0) {
        const int code = ~cur;
        const int first = code & 0x0fffffff;
        const int cnt = (code >> 28) + 1;
        for (int e = 0; e < cnt; e++) {
            const int k = first + e;
            if (k == (ray.self_k ^ RZ_SELF_OUT)) continue;   // left outward: cannot be hit again
            const float4 s = __ldg(a.set.cr + k);
            const float4 v = __ldg(a.set.vel + k);
            if (STATS) c_sph++;
            float nb, nd;   // the one sphere test of the backend (rz_device.cuh): bit-identical to the packed searches
            rz_sphere_test(s.x, s.y, s.z, v.x, v.y, v.z, s.w, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, ray.time, nb, nd);
            if (nd < 0.0f) rz_consider(k, nb, nd, ray.self_k, a.t_min, bt, bk);
        }
        cur = sp > 0 ? stack[--sp] : RZ_SENTINEL;
    }
}

// LIST (not with QUEUE): the adaptive rounds' form, paths of the pixels a.px_list names (RzPathArgs::px_list).
template <bool STATS, bool QUEUE, int UNIT = 512, bool LIST = false, int SOBOL = 0>
__global__ void __launch_bounds__(128, RZ_BVH_MINB) rz_bvh_kernel(const RzPathArgs a) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const float4 *__restrict__ nodes = reinterpret_cast<const float4 *>(a.bvh);

    // warp-uniform work-unit state (as in rz_path_kernel)
    bool have_unit = true;
    uint32_t unit_lp0 = 0, unit_s0 = 0, unit_paths = 0, k_next = 0;
    const uint32_t n_entries = QUEUE ? min(*a.q_in_count, a.queue_cap) : 0u;   // QUEUE: paths start from queue entries
    // ... in units of UNIT entries: 512 when the queue holds every path of a pass (a large scene's job after the camera stage), 64
    // as the tail of the staged K1 — ~2 M entries per pass, less than one 512-entry unit per resident warp: the launch then lasts
    // as long as ONE warp needs for 512 paths while most warps hold nothing (tail of a serial-pass config-2 render: 4.7 -> 3.5 ms).
    // A unit boundary costs one atomic; the lanes refill across it.  (A unit size computed from the queue length on the device
    // did the same for the tail but cost the large-scene case 1.4 %: one more live value at the 64-register cap.)
    constexpr uint32_t unit_size = (uint32_t)UNIT;
    const uint32_t n_units = QUEUE ? (n_entries + unit_size - 1u) / unit_size : a.n_units;

    // per-lane path state
    RzRay ray;
    ray.o = f3(0.f, 0.f, 0.f); ray.d = f3(0.f, 1.f, 0.f); ray.time = 0.f; ray.self_k = -1;
    float3 thr = f3(0.f, 0.f, 0.f);
    uint32_t lp = 0, gpix = 0, sample = 0, seg = 0;
    bool alive = false;
    // per-lane traversal state
    int cur = RZ_SENTINEL, sp = 0, bk = -1;
    float bt = 3.0e38f, ix = 0.f, iy = 0.f, iz = 0.f;
    int stack[RZ_STACK];

    unsigned long long c_paths = 0, c_segs = 0, c_nodes = 0, c_sph = 0, c_hit[3] = {0, 0, 0}, c_sky = 0, c_abs = 0, c_depth = 0;

    const int descend_min = (int)a.bvh_descend_min;
    auto start_traversal = [&]() {
        ix = 1.0f / ray.d.x; iy = 1.0f / ray.d.y; iz = 1.0f / ray.d.z;
        bt = 3.0e38f; bk = -1; sp = 0; cur = 0;
    };

    while (true) {
        // ------------------------------------------------------------ shade finished traversals
        if (alive && cur == RZ_SENTINEL) {
            if (STATS) c_segs++;
            uint32_t kind;
            const int res = rz_shade_segment(a, ray, thr, seg, lp, gpix, sample, bk, kind, SOBOL);
            if (STATS) {
                if (kind < 3u) c_hit[kind]++;
                if (res == RZ_END_SKY) c_sky++;
                if (res == RZ_END_ABSORBED) c_abs++;
                if (res == RZ_END_DEPTH) c_depth++;
            }
            if (res != RZ_CONT) alive = false; else start_traversal();
        }
        // ------------------------------------------------------------ regenerate dead lanes
        {
            bool need = !alive;
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
                        unit_lp0 = u * unit_size;                  // first queue entry of the unit
                        unit_paths = min(unit_size, n_entries - unit_lp0);
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
                        ray.o = f3(qa.x, qa.y, qa.z); ray.time = qa.w;
                        ray.d = f3(qb.x, qb.y, qb.z); ray.self_k = __float_as_int(qb.w);
                        if (a.self_map && ray.self_k >= 0)                                          // entry written by a brute-force stage
                            ray.self_k = a.self_map[ray.self_k & ~RZ_SELF_OUT] | (ray.self_k & RZ_SELF_OUT);
                        thr = f3(qc.x, qc.y, qc.z); seg = __float_as_uint(qc.w);
                        lp = __float_as_uint(qd.x); gpix = __float_as_uint(qd.y); sample = __float_as_uint(qd.z);
                        alive = true;
                        start_traversal();
                        need = false;
                    } else {
                        uint32_t nlp = unit_lp0 + (k & 31u);
                        if (nlp < (LIST ? a.n_list : a.n_local_px)) {
                            if (LIST) nlp = __ldg(a.px_list + nlp);
                            uint32_t pi, pj;
                            rz_local_to_global(nlp, a.width, a.shard_index, a.shard_count, a.band_rows, pi, pj);
                            lp = nlp;
                            gpix = pj * a.width + pi;
                            sample = a.sample_offset + unit_s0 + (k >> 5);
                            ray = rz_camera_ray(a.cam, pi, pj, gpix, sample, a.seed_lo, a.seed_hi, SOBOL);
                            thr = f3(1.f, 1.f, 1.f);
                            seg = 0;
                            alive = a.max_depth > 0u;
                            if (STATS) { c_paths++; if (!alive) c_depth++; }
                            if (alive) start_traversal();
                            need = !alive;
                        }
                    }
                }
                k_next += min((uint32_t)__popc(mask), avail);
            }
        }
        if (!__any_sync(0xffffffffu, alive)) break;

        // ------------------------------------------------------------ traversal burst
        // keep stepping while enough lanes are busy; once work has run out, drain completely
        const int active_min = have_unit ? (int)a.bvh_active_min : 1;
        while (__popc(__ballot_sync(0xffffffffu, cur != RZ_SENTINEL)) >= active_min) {
            rz_bvh_round<STATS>(a, nodes, ray, ix, iy, iz, cur, sp, stack, bt, bk, descend_min, c_nodes, c_sph);
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

// Staged form for large jobs on large scenes: the first segments of every path are traced one segment per launch, camera
// rays tile by tile and scattered rays in SORTED order (key of rz_sort_key: origin cell, octant, reach), 32 rays per warp at
// a time.  Rays that start together and head the same way walk the same nodes, so the warp stays converged and the nodes stay
// in L1; survivors go to the next queue, and the tail of the paths to the persistent kernel above (QUEUE).
// CAMERA: the camera rays of a work unit — an 8 x 4-pixel block x `chunk` samples — do not walk the tree one by one; the warp
// culls the tree once against the block's cone and the rays search the surviving spheres as a list (below).  The sorted stages (CAMERA = false) are off by default (RzTuning::bvh_stages = 0: measured as a loss).
template <bool STATS, bool CAMERA, int SOBOL = 0>
__global__ void __launch_bounds__(128, CAMERA ? RZ_BVH_CAMERA_MINB : RZ_BVH_MINB) rz_bvh_stage_kernel(const RzPathArgs a) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const float4 *__restrict__ nodes = reinterpret_cast<const float4 *>(a.bvh);
    const uint32_t n_in = CAMERA ? 0u : min(*a.q_in_count, a.queue_cap);
    const uint32_t ue = a.unit_entries;
    const uint32_t n_units = CAMERA ? a.n_units : (n_in + ue - 1u) / ue;
    const int descend_min = (int)a.bvh_descend_min;
    int stack[RZ_STACK];
    unsigned long long c_paths = 0, c_segs = 0, c_nodes = 0, c_sph = 0, c_hit[3] = {0, 0, 0}, c_sky = 0, c_abs = 0, c_depth = 0;
    // per-warp scratch of the camera stage's tile lists: candidate spheres (stationary ones from the front, moving ones from the
    // back), their positions in the set, the cull's ring buffer of nodes; idl = 0, 1, 2, ... (the lists the packed search walks)
    __shared__ float4 s_cl_cr[CAMERA ? 4 : 1][CAMERA ? RZ_CL_CAP : 1], s_cl_vel[CAMERA ? 4 : 1][CAMERA ? RZ_CL_CAP : 1];
    __shared__ int s_cl_gid[CAMERA ? 4 : 1][CAMERA ? RZ_CL_CAP : 1], s_cl_wl[CAMERA ? 4 : 1][CAMERA ? RZ_CL_WL : 1];
    __shared__ unsigned short s_cl_idl[CAMERA ? RZ_CL_CAP : 1];
    if (CAMERA) {
        for (unsigned i = threadIdx.x; i < (unsigned)RZ_CL_CAP; i += blockDim.x) s_cl_idl[i] = (unsigned short)i;
        __syncthreads();
    }

    while (true) {
        unsigned u = 0;
        if (lane == 0) u = atomicAdd(a.unit_counter, 1u);
        u = __shfl_sync(0xffffffffu, u, 0);
        if (u >= n_units) break;
        uint32_t n_batches, pi = 0, pj = 0, lp0 = 0, gpix0 = 0, s0 = 0, e0 = 0, ne = 0;
        bool valid = true;
        if (CAMERA) {
            u += a.unit_base;
            const uint32_t tile = u / a.n_chunks, chunk = u - tile * a.n_chunks;
            if (a.tile_w) {   // 8 x 4 pixel blocks (the host sets tile_w = 8 for the BVH family and counts the units accordingly)
                const uint32_t tiles_x = (a.width + 7u) >> 3;
                const uint32_t ty = tile / tiles_x, tx = tile - ty * tiles_x;
                const uint32_t ti = tx * 8u + (lane & 7u), tr = ty * 4u + (lane >> 3);
                lp0 = tr * a.width + ti;
                valid = ti < a.width && lp0 < a.n_local_px;
            } else {
                lp0 = tile * 32u + lane;
                valid = lp0 < a.n_local_px;
            }
            if (valid) rz_local_to_global(lp0, a.width, a.shard_index, a.shard_count, a.band_rows, pi, pj);
            gpix0 = pj * a.width + pi;
            s0 = chunk * a.chunk;
            n_batches = min(a.chunk, a.spp - s0);
        } else {
            e0 = u * ue; ne = min(ue, n_in - e0);
            n_batches = (ne + 31u) / 32u;
        }
        if (CAMERA) {
            // ---- Camera rays of a 32-pixel tile are coherent: instead of 32 x chunk separate walks, the warp culls the TREE once
            // against the tile's cone (rz_tile_cone / rz_tile_keep of the primary kernel; a child box enters as its bounding
            // sphere, which the per-sphere test cannot pass where the box's does not) and the tile's rays then search the
            // surviving spheres as a list, two rays per lane packed into FP32x2 (rz_search_lists_r2: the arithmetic of every
            // other search, the same (t, k)).  Breadth first, up to 32 nodes per step, one lane per node.  A tile whose list or
            // frontier outgrows its scratch (the horizon band of a large scene) falls through to the per-ray walk below.
            const unsigned warp = threadIdx.x >> 5;
            float4 *w_cr = s_cl_cr[warp], *w_vel = s_cl_vel[warp];
            int *w_gid = s_cl_gid[warp], *w_wl = s_cl_wl[warp];
            int n_s = 0, n_m = 0;
            bool lists_ok = true;
            {
                const float3 pc = rz_tile_pixel_dir(a.cam, pi, pj);
                float3 ax = valid ? normalize3(pc) : f3(0.f, 0.f, 0.f);
                for (int o = 16; o > 0; o >>= 1) {
                    ax.x += __shfl_xor_sync(0xffffffffu, ax.x, o); ax.y += __shfl_xor_sync(0xffffffffu, ax.y, o); ax.z += __shfl_xor_sync(0xffffffffu, ax.z, o);
                }
                const bool has_axis = rz_tile_axis(ax);
                float cmin = valid ? rz_tile_corner_cos(a.cam, pc, ax) : 1.0f;
                for (int o = 16; o > 0; o >>= 1) cmin = fminf(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
                const RzTileCone cone = rz_tile_cone(a.cam, ax, has_axis, cmin, a.focus_dist, a.lens_radius);
                unsigned head = 0u, tail = 1u;
                __syncwarp();
                if (lane == 0) w_wl[0] = 0;   // the root
                __syncwarp();
                while (head < tail && lists_ok) {
                    const unsigned take = min(32u, tail - head);
                    bool keep[2] = {false, false};
                    int ref[2] = {0, 0};
                    if (lane < take) {
                        const int node = w_wl[(head + lane) & (unsigned)(RZ_CL_WL - 1)];
                        const float4 q0 = __ldg(nodes + node * 4 + 0), q1 = __ldg(nodes + node * 4 + 1), q2 = __ldg(nodes + node * 4 + 2);   // lo0 lo1 hi0 hi1 per axis
                        const int4 q3 = __ldg(reinterpret_cast<const int4 *>(nodes + node * 4 + 3));
                        if (STATS) c_nodes += 2;
                        keep[0] = rz_tile_keep_box(cone, q0.x, q0.z, q1.x, q1.z, q2.x, q2.z);
                        keep[1] = rz_tile_keep_box(cone, q0.y, q0.w, q1.y, q1.w, q2.y, q2.w);
                        ref[0] = q3.x; ref[1] = q3.y;
                    }
                    head += take;
                    // internal children join the frontier
                    const bool p0 = keep[0] && ref[0] >= 0, p1 = keep[1] && ref[1] >= 0;
                    const unsigned m0 = __ballot_sync(0xffffffffu, p0), m1 = __ballot_sync(0xffffffffu, p1);
                    const unsigned n0 = (unsigned)__popc(m0), n1 = (unsigned)__popc(m1);
                    if (tail + n0 + n1 - head > (unsigned)RZ_CL_WL) { lists_ok = false; break; }
                    if (p0) w_wl[(tail + (unsigned)__popc(m0 & lt_mask)) & (unsigned)(RZ_CL_WL - 1)] = ref[0];
                    if (p1) w_wl[(tail + n0 + (unsigned)__popc(m1 & lt_mask)) & (unsigned)(RZ_CL_WL - 1)] = ref[1];
                    tail += n0 + n1;
                    // leaf children: their spheres, each against the cone with its own radius and motion
#pragma unroll 1
                    for (int c = 0; c < 2 && lists_ok; c++) {
                        const bool leaf = keep[c] && ref[c] < 0;
                        const int code = ~ref[c];
                        const int first = code & 0x0fffffff;
                        const int lc = leaf ? (code >> 28) + 1 : 0;
#pragma unroll 1
                        for (int e = 0; e < 8; e++) {
                            const bool has = e < lc;
                            if (!__any_sync(0xffffffffu, has)) break;
                            const int k = first + e;
                            float4 S = make_float4(0.f, 0.f, 0.f, 1.f), V = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (has) { S = __ldg(a.set.cr + k); V = __ldg(a.set.vel + k); }
                            const bool kp = has && rz_tile_keep(cone, S.x, S.y, S.z, V.x, V.y, V.z, S.w);
                            const bool still = V.x == 0.f && V.y == 0.f && V.z == 0.f;
                            const unsigned ms = __ballot_sync(0xffffffffu, kp && still), mm = __ballot_sync(0xffffffffu, kp && !still);
                            if (n_s + n_m + __popc(ms) + __popc(mm) > RZ_CL_CAP) { lists_ok = false; break; }
                            if (kp && still) { const int i = n_s + __popc(ms & lt_mask); w_cr[i] = S; w_gid[i] = k; }
                            if (kp && !still) { const int i = RZ_CL_CAP - 1 - (n_m + __popc(mm & lt_mask)); w_cr[i] = S; w_vel[i] = V; w_gid[i] = k; }
                            n_s += __popc(ms); n_m += __popc(mm);
                        }
                    }
                    __syncwarp();
                }
            }
            __syncwarp();
            if (lists_ok) {
                const unsigned short *ls = s_cl_idl, *lm = s_cl_idl + (RZ_CL_CAP - n_m);
#pragma unroll 1
                for (uint32_t b = 0; b < n_batches; b += 2u) {
                    RzRay rays[2];
                    bool live[2];
                    uint32_t smp[2];
#pragma unroll
                    for (int r = 0; r < 2; r++) {
                        smp[r] = a.sample_offset + s0 + b + (uint32_t)r;
                        const bool have = valid && (b + (uint32_t)r < n_batches);
                        live[r] = have && a.max_depth > 0u;
                        if (STATS && have) { c_paths++; if (!live[r]) c_depth++; }
                        if (live[r]) rays[r] = rz_camera_ray(a.cam, pi, pj, gpix0, smp[r], a.seed_lo, a.seed_hi, SOBOL);
                        else { rays[r].o = f3(0.f, 0.f, 0.f); rays[r].d = f3(0.f, 1.f, 0.f); rays[r].time = 0.f; rays[r].self_k = -1; }
                    }
                    float bt[2] = {3.0e38f, 3.0e38f};
                    int bk[2] = {-1, -1};
                    rz_search_lists_r2(w_cr, w_vel, ls, n_s, lm, n_m, rays, a.t_min, bt, bk);
                    if (STATS) c_sph += (unsigned long long)(n_s + n_m) * ((live[0] ? 1u : 0u) + (live[1] ? 1u : 0u));
                    float3 thr[2] = {f3(1.f, 1.f, 1.f), f3(1.f, 1.f, 1.f)};
                    uint32_t seg[2] = {0u, 0u};
                    bool cont[2] = {false, false};
                    // one copy of the shading code for both rays (code size: DESIGN.md section 3): shade slot 0, exchange, shade again, exchange back
#pragma unroll 1
                    for (int trip = 0; trip < 2; trip++) {
                        if (live[0]) {
                            const int hit = bk[0] < 0 ? -1 : (w_gid[bk[0] & ~RZ_FAR_BIT] | (bk[0] & RZ_FAR_BIT));   // list slot -> position in the set
                            if (STATS) c_segs++;
                            uint32_t kind;
                            const int res = rz_shade_segment(a, rays[0], thr[0], seg[0], lp0, gpix0, smp[0], hit, kind, SOBOL);
                            if (STATS) {
                                if (kind < 3u) c_hit[kind]++;
                                if (res == RZ_END_SKY) c_sky++;
                                if (res == RZ_END_ABSORBED) c_abs++;
                                if (res == RZ_END_DEPTH) c_depth++;
                            }
                            cont[0] = res == RZ_CONT;
                        }
                        { const RzRay t = rays[0]; rays[0] = rays[1]; rays[1] = t; }
                        { const float3 t = thr[0]; thr[0] = thr[1]; thr[1] = t; }
                        { const uint32_t t = seg[0]; seg[0] = seg[1]; seg[1] = t; }
                        { const uint32_t t = smp[0]; smp[0] = smp[1]; smp[1] = t; }
                        { const int t = bk[0]; bk[0] = bk[1]; bk[1] = t; }
                        { const bool t = live[0]; live[0] = live[1]; live[1] = t; }
                        { const bool t = cont[0]; cont[0] = cont[1]; cont[1] = t; }
                    }
                    const uint32_t lp2[2] = {lp0, lp0}, gp2[2] = {gpix0, gpix0};
                    rz_queue_push2(a, cont, lane, lt_mask, rays, thr, seg, lp2, gp2, smp);
                }
                continue;   // next unit
            }
        }
        for (uint32_t b = 0; b < n_batches; b++) {
            RzRay ray;
            float3 thr = f3(1.f, 1.f, 1.f);
            uint32_t seg = 0, lp = lp0, gpix = gpix0, smp = 0;
            bool live;
            if (CAMERA) {
                smp = a.sample_offset + s0 + b;
                live = valid && a.max_depth > 0u;
                if (STATS && valid) { c_paths++; if (!live) c_depth++; }
                if (live) ray = rz_camera_ray(a.cam, pi, pj, gpix, smp, a.seed_lo, a.seed_hi, SOBOL);
            } else {
                const uint32_t i = b * 32u + lane;
                live = i < ne;
                if (live) {
                    const float4 *e = a.q_in + (size_t)(a.q_in_idx[e0 + i] & RZ_IDX_MASK) * 4u;
                    const float4 qa = __ldcs(e), qb = __ldcs(e + 1), qc = __ldcs(e + 2), qd = __ldcs(e + 3);
                    ray.o = f3(qa.x, qa.y, qa.z); ray.time = qa.w;
                    ray.d = f3(qb.x, qb.y, qb.z); ray.self_k = __float_as_int(qb.w);
                    thr = f3(qc.x, qc.y, qc.z); seg = __float_as_uint(qc.w);
                    lp = __float_as_uint(qd.x); gpix = __float_as_uint(qd.y); smp = __float_as_uint(qd.z);
                }
            }
            if (!live) { ray.o = f3(0.f, 0.f, 0.f); ray.d = f3(0.f, 1.f, 0.f); ray.time = 0.f; ray.self_k = -1; }
            const float ix = 1.0f / ray.d.x, iy = 1.0f / ray.d.y, iz = 1.0f / ray.d.z;
            float bt = 3.0e38f;
            int bk = -1, sp = 0, cur = live ? 0 : RZ_SENTINEL;
            while (__any_sync(0xffffffffu, cur != RZ_SENTINEL))
                rz_bvh_round<STATS>(a, nodes, ray, ix, iy, iz, cur, sp, stack, bt, bk, descend_min, c_nodes, c_sph);
            bool cont = false;
            if (live) {
                if (STATS) c_segs++;
                uint32_t kind;
                const int res = rz_shade_segment(a, ray, thr, seg, lp, gpix, smp, bk, kind, SOBOL);
                if (STATS) {
                    if (kind < 3u) c_hit[kind]++;
                    if (res == RZ_END_SKY) c_sky++;
                    if (res == RZ_END_ABSORBED) c_abs++;
                    if (res == RZ_END_DEPTH) c_depth++;
                }
                cont = res == RZ_CONT;
            }
            rz_queue_push(a, cont, lane, lt_mask, ray, thr, seg, lp, gpix, smp);
        }
    }

    if (STATS) {
        unsigned long long v[10] = {c_paths, c_segs, c_sph, c_nodes, c_hit[0], c_hit[1], c_hit[2], c_sky, c_abs, c_depth};
#pragma unroll
        for (int i = 0; i < 10; i++) {
            unsigned long long sum = v[i];
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            if (lane == 0 && sum) atomicAdd(&a.stats->v[i], sum);
        }
    }
}

// First-hit albedo of a guide sample: the attenuation rz_scatter gives for the hit (rz_shade_segment's decode of the material
// record, kept apart so that the path kernels stay as they are), whether or not a metal's scatter would be absorbed.
__device__ __forceinline__ float3 rz_guide_albedo(const RzPathArgs &a, int k, const RzHit &h) {
    const float4 *mr = a.mats.rec + 4u * a.set.mat[k];
    const float4 m0 = __ldg(mr);
    const uint32_t mbits = __float_as_uint(m0.x);
    if ((mbits & 3u) >= 2u) return f3(1.f, 1.f, 1.f);   // dielectric (rz_scatter's third branch)
    const float4 m1 = __ldg(mr + 1), m2 = __ldg(mr + 2), m3 = __ldg(mr + 3);
    RzMatRec M;
    M.kind = mbits & 3u; M.method = (mbits >> 2) & 3u; M.solid = ((mbits >> 4) & 1u) != 0u; M.checker2 = ((mbits >> 5) & 1u) != 0u;
    M.fuzz = m0.y; M.ior = m0.z; M.tex = __float_as_uint(m0.w);
    M.color = f3(m1.x, m1.y, m1.z); M.odd = f3(m2.x, m2.y, m2.z);
    M.inv_scale = __hiloint2double(__float_as_int(m3.y), __float_as_int(m3.x));
    return M.solid ? M.color : M.checker2 ? rz_checker2(M, h.px, h.py, h.pz) : rz_texture(a.texs, M.tex, h.px, h.py, h.pz);
}

// Guide buffers: the camera samples [sample_offset, sample_offset + spp) of every local pixel, each traced to its first hit by
// the unstaged K3's walk (rz_bvh_round, the same tree and the same (t, k)), in this translation unit so that the camera ray
// and the walk compile with the path kernels' flags.  One warp per 8 x 4 block of local rows, one lane per pixel, the warp's
// samples in lockstep: a block's rays fan out over a third of the angle of 32 pixels of a row (the camera stage's reason for
// the same blocks), so the lanes visit more of the same nodes.  Each lane sums its pixel's samples in f64, in sample order, and
// divides once: the result depends on (scene, camera, seed, pixel, sample range) only.
template <int SOBOL>
__global__ void __launch_bounds__(128, RZ_BVH_MINB) rz_guides_kernel(const RzGuideArgs g) {
    const RzPathArgs &a = g.a;
    const unsigned lane = threadIdx.x & 31u;
    const float4 *__restrict__ nodes = reinterpret_cast<const float4 *>(a.bvh);
    const uint32_t block = blockIdx.x * 4u + (threadIdx.x >> 5), tiles_x = (a.width + 7u) >> 3;
    const uint32_t ty = block / tiles_x, tx = block - ty * tiles_x;
    const uint32_t ti = tx * 8u + (lane & 7u), lp = (ty * 4u + (lane >> 3)) * a.width + ti;
    const bool valid = ti < a.width && lp < a.n_local_px;
    if (!__any_sync(0xffffffffu, valid)) return;   // the grid's last CTA: a warp past the last block
    uint32_t pi = 0, pj = 0;
    if (valid) rz_local_to_global(lp, a.width, a.shard_index, a.shard_count, a.band_rows, pi, pj);
    const uint32_t gpix = pj * a.width + pi;
    const int descend_min = (int)a.bvh_descend_min;
    int stack[RZ_STACK];
    unsigned long long c_none = 0;   // rz_bvh_round's counters: untouched without STATS
    double alb_r = 0, alb_g = 0, alb_b = 0, nx = 0, ny = 0, nz = 0, dist = 0;
    uint32_t hits = 0;
    for (uint32_t s = 0; s < a.spp; s++) {
        RzRay ray;
        if (valid) ray = rz_camera_ray(a.cam, pi, pj, gpix, a.sample_offset + s, a.seed_lo, a.seed_hi, SOBOL);
        else { ray.o = f3(0.f, 0.f, 0.f); ray.d = f3(0.f, 1.f, 0.f); ray.time = 0.f; ray.self_k = -1; }
        const float ix = 1.0f / ray.d.x, iy = 1.0f / ray.d.y, iz = 1.0f / ray.d.z;
        float bt = 3.0e38f;
        int bk = -1, sp = 0, cur = valid ? 0 : RZ_SENTINEL;
        while (__any_sync(0xffffffffu, cur != RZ_SENTINEL))
            rz_bvh_round<false>(a, nodes, ray, ix, iy, iz, cur, sp, stack, bt, bk, descend_min, c_none, c_none);
        if (!valid) continue;
        float3 alb;
        if (bk < 0) {
            alb = rz_sky(ray.d);   // a miss guides to its own radiance
        } else {
            const int k = bk & ~RZ_FAR_BIT;
            const RzHit h = rz_refine_hit(a.set, ray, k, (bk & RZ_FAR_BIT) != 0);
            alb = rz_guide_albedo(a, k, h);
            nx += (double)h.n.x; ny += (double)h.n.y; nz += (double)h.n.z;
            dist += (double)bt;
            hits++;
        }
        alb_r += (double)alb.x; alb_g += (double)alb.y; alb_b += (double)alb.z;
    }
    if (!valid) return;
    size_t dst = lp;
    if (g.dev_count > 1u) {   // rz_resolve_kernel's band arithmetic
        const uint32_t lr = lp / a.width, lb = lr / a.band_rows, within = lr - lb * a.band_rows;
        dst = (size_t)((lb * g.dev_count + g.dev_index) * a.band_rows + within) * a.width + ti;
    }
    const double n = (double)a.spp;
    if (g.out_albedo) g.out_albedo[dst] = make_float4((float)(alb_r / n), (float)(alb_g / n), (float)(alb_b / n), (float)((double)hits / n));
    if (g.out_normal)
        g.out_normal[dst] = make_float4((float)(nx / n), (float)(ny / n), (float)(nz / n), hits ? (float)(dist / (double)hits) : 0.f);
}

// inst: the kernel's instances (rz_pick_instance), launched on the persistent grid
template <class F>
cudaError_t launch_kernel(F inst, const RzPathArgs &a, int collect_stats, int sm_count, cudaStream_t stream) {
    const auto kern = rz_pick_instance(a, collect_stats, inst);
    int grid = 0;
    const cudaError_t e = rz_persistent_grid(kern, 0, sm_count, &grid);
    if (e != cudaSuccess) return e;
    kern<<<grid, 128, 0, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace

extern "C" cudaError_t rz_bvh_warm(void) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, rz_bvh_kernel<false, false>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, rz_bvh_stage_kernel<false, true>);
    return e;
}

static void rz_bvh_tuning(RzPathArgs &b) {   // defaults are the measured optimum (file header); RzTuning overrides them
    if (b.bvh_active_min < 1u) b.bvh_active_min = 8u;
    if (b.bvh_active_min > 32u) b.bvh_active_min = 32u;
    if (b.bvh_descend_min < 1u) b.bvh_descend_min = 24u;
    if (b.stack_cap < 1u || b.stack_cap > (uint32_t)RZ_STACK) b.stack_cap = (uint32_t)RZ_STACK;
}

// The persistent kernel: whole paths from the camera (q_in == nullptr; only the pixels of px_list when it is set) or the tails
// of paths from a queue.
extern "C" cudaError_t rz_launch_bvh(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream) {
    RzPathArgs b = *a;
    rz_bvh_tuning(b);
    if (b.q_in && b.self_map)   // the tail of the staged K1 (entries written by a brute-force stage): a short queue, small units
        return launch_kernel([](auto S, auto M) { return rz_bvh_kernel<decltype(S)::value, true, 64, false, decltype(M)::value>; }, b, collect_stats, sm_count, stream);
    if (b.q_in)
        return launch_kernel([](auto S, auto M) { return rz_bvh_kernel<decltype(S)::value, true, 512, false, decltype(M)::value>; }, b, collect_stats, sm_count, stream);
    if (b.px_list)
        return launch_kernel([](auto S, auto M) { return rz_bvh_kernel<decltype(S)::value, false, 512, true, decltype(M)::value>; }, b, collect_stats, sm_count, stream);
    return launch_kernel([](auto S, auto M) { return rz_bvh_kernel<decltype(S)::value, false, 512, false, decltype(M)::value>; }, b, collect_stats, sm_count, stream);
}

// Guide buffers of the device's local pixels: one warp per 8 x 4 block, four per CTA.
extern "C" cudaError_t rz_launch_guides(const RzGuideArgs *g, cudaStream_t stream) {
    RzGuideArgs b = *g;
    rz_bvh_tuning(b.a);
    const uint32_t rows = b.a.width ? b.a.n_local_px / b.a.width : 0u;
    const uint32_t blocks = ((b.a.width + 7u) / 8u) * ((rows + 3u) / 4u);
    if (blocks == 0u) return cudaSuccess;
    rz_pick_instance(b.a, 0, [](auto, auto M) { return rz_guides_kernel<decltype(M)::value>; })<<<(blocks + 3u) / 4u, 128, 0, stream>>>(b);
    return cudaGetLastError();
}

// One segment per launch: camera segments (q_in == nullptr) or the sorted entries of q_in; survivors -> q_out.
extern "C" cudaError_t rz_launch_bvh_stage(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream) {
    RzPathArgs b = *a;
    rz_bvh_tuning(b);
    if (!b.q_in)
        return launch_kernel([](auto S, auto M) { return rz_bvh_stage_kernel<decltype(S)::value, true, decltype(M)::value>; }, b, collect_stats, sm_count, stream);
    return launch_kernel([](auto S, auto M) { return rz_bvh_stage_kernel<decltype(S)::value, false, decltype(M)::value>; }, b, collect_stats, sm_count, stream);
}
