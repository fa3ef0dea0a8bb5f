// rz_search.cuh — device-only pieces shared by the megakernel (rz_path.cu) and the wavefront
// kernels (rz_wavefront.cu): bulk-copy/mbarrier PTX helpers, the closest-hit searches and the
// per-segment shading step.  Both kernel families call the SAME functions, so for equal RNG keys
// they produce bit-identical radiance.
#pragma once
#include <type_traits>

#include "rz_device.cuh"


// ------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t rz_smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void rz_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(rz_smem_addr(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void rz_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(rz_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void rz_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(rz_smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(rz_smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void rz_mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(rz_smem_addr(bar)), "r"(parity)
            : "memory");
    }
}

// ------------------------------------------------------------------------------ K1 search, packed
// rz_sphere_test (rz_device.cuh) issued as Blackwell packed-FP32 instructions (PTX add/mul/fma.rn.f32x2 -> SASS FADD2 /
// FMUL2 / FFMA2): one instruction works on TWO SPHERES (the .x/.y halves of a 64-bit register pair) against one ray, whose
// operands enter as 32-bit broadcast registers (`R.F32` in SASS), so rays cost no extra registers.  Per ray and sphere PAIR:
//   stationary: 3 FADD2 (oc) + FMUL2 + 2 FFMA2 (nb) + 3 FFMA2 (l) + 3 FFMA2 (nd) = 12 issue slots for 2 tests
//   moving    : + 3 FFMA2 for centre(t) = c0 + v * time (geom.zig:40)              = 15 issue slots
// Every half follows the operation order of rz_sphere_test exactly (IEEE rn, FTZ): bit-identical (t, k) in every search.
// s_pk: pair-interleaved sphere set in shared memory (layout: RzSphereSet::pk).
__device__ __forceinline__ float2 rz_f2(float x, float y) { return make_float2(x, y); }

// the ray's operands as the packed test wants them: -o (so that C - o is an add) and -d (so that nb needs no negation)
struct RzRayOps {
    float nox, noy, noz, ndx, ndy, ndz, dx, dy, dz, time;
};
__device__ __forceinline__ RzRayOps rz_ray_ops(const RzRay &r) {
    RzRayOps q;
    q.nox = -r.o.x; q.noy = -r.o.y; q.noz = -r.o.z;
    q.ndx = -r.d.x; q.ndy = -r.d.y; q.ndz = -r.d.z;
    q.dx = r.d.x; q.dy = r.d.y; q.dz = r.d.z;
    q.time = r.time;
    return q;
}

// two stationary spheres (A = cx0 cx1 cy0 cy1, B = cz0 cz1 w0 w1) against one ray
__device__ __forceinline__ void rz_test2_static(const float4 A, const float4 B, const RzRayOps &q, float2 &nb, float2 &nd) {
    const float2 ocx = __fadd2_rn(rz_f2(A.x, A.y), rz_f2(q.nox, q.nox));
    const float2 ocy = __fadd2_rn(rz_f2(A.z, A.w), rz_f2(q.noy, q.noy));
    const float2 ocz = __fadd2_rn(rz_f2(B.x, B.y), rz_f2(q.noz, q.noz));
    nb = __ffma2_rn(ocz, rz_f2(q.ndz, q.ndz), __ffma2_rn(ocy, rz_f2(q.ndy, q.ndy), __fmul2_rn(ocx, rz_f2(q.ndx, q.ndx))));
    const float2 lx = __ffma2_rn(nb, rz_f2(q.dx, q.dx), ocx), ly = __ffma2_rn(nb, rz_f2(q.dy, q.dy), ocy), lz = __ffma2_rn(nb, rz_f2(q.dz, q.dz), ocz);
    nd = __ffma2_rn(lz, lz, __ffma2_rn(ly, ly, __ffma2_rn(lx, lx, rz_f2(B.z, B.w))));
}

// two moving spheres (+ VA = vx0 vx1 vy0 vy1, VB = vz0 vz1 . .).  oc = (c0 - o) + v * time: each instruction reads ONE register
// pair that came from shared memory (two "cold" 64-bit sources cost an FFMA2 ~3.3 cycles instead of 2)
__device__ __forceinline__ void rz_test2_moving(const float4 A, const float4 B, const float4 VA, const float4 VB, const RzRayOps &q, float2 &nb,
                                                float2 &nd) {
    const float2 tm = rz_f2(q.time, q.time);
    const float2 ocx = __ffma2_rn(rz_f2(VA.x, VA.y), tm, __fadd2_rn(rz_f2(A.x, A.y), rz_f2(q.nox, q.nox)));
    const float2 ocy = __ffma2_rn(rz_f2(VA.z, VA.w), tm, __fadd2_rn(rz_f2(A.z, A.w), rz_f2(q.noy, q.noy)));
    const float2 ocz = __ffma2_rn(rz_f2(VB.x, VB.y), tm, __fadd2_rn(rz_f2(B.x, B.y), rz_f2(q.noz, q.noz)));
    nb = __ffma2_rn(ocz, rz_f2(q.ndz, q.ndz), __ffma2_rn(ocy, rz_f2(q.ndy, q.ndy), __fmul2_rn(ocx, rz_f2(q.ndx, q.ndx))));
    const float2 lx = __ffma2_rn(nb, rz_f2(q.dx, q.dx), ocx), ly = __ffma2_rn(nb, rz_f2(q.dy, q.dy), ocy), lz = __ffma2_rn(nb, rz_f2(q.dz, q.dz), ocz);
    nd = __ffma2_rn(lz, lz, __ffma2_rn(ly, ly, __ffma2_rn(lx, lx, rz_f2(B.z, B.w))));
}

// Brute force over the whole set (RZ_VARIANT_MEGA_SINGLE, the wavefront's intersect stage, the brute-force tail).
// G2 = sphere pairs per loop iteration (2 => 8 tests of 2 rays share one min tree + branch).  Sphere operands are warp-uniform
// LDS.128 broadcasts; only when some lane has nd < 0 does the warp enter the rare path (rz_consider: square root, root rule).
// Measured and not adopted: operands from the constant bank through the uniform datapath, the moving loop unrolled by 2
// (1475 vs 1519 Mpaths/s) and a warp-uniform entry into the rare path, __any_sync (no difference).
template <int R, int G2>
__device__ __forceinline__ void rz_search_brute2(const float4 *__restrict__ src, int n_static_pad, int n_pad,
                                                 const RzRay (&ray)[R], float t_min, float (&bt)[R], int (&bk)[R]) {
    RzRayOps q[R];
#pragma unroll
    for (int r = 0; r < R; r++) q[r] = rz_ray_ops(ray[r]);
    int f = 0;   // float4 index into the pair-interleaved set
    int k = 0;
#pragma unroll 1
    for (; k < n_static_pad; k += 2 * G2, f += 2 * G2) {
        float4 A[G2], B[G2];
#pragma unroll
        for (int j = 0; j < G2; j++) { A[j] = src[f + 2 * j]; B[j] = src[f + 2 * j + 1]; }
        float2 nb[R][G2], nd[R][G2];
        float m = 1.0f;
#pragma unroll
        for (int r = 0; r < R; r++) {
#pragma unroll
            for (int j = 0; j < G2; j++) {
                rz_test2_static(A[j], B[j], q[r], nb[r][j], nd[r][j]);
                m = fminf(m, fminf(nd[r][j].x, nd[r][j].y));
            }
        }
        if (m < 0.0f) {
#pragma unroll
            for (int r = 0; r < R; r++)
#pragma unroll
                for (int j = 0; j < G2; j++) {
                    if (nd[r][j].x < 0.0f) rz_consider(k + 2 * j, nb[r][j].x, nd[r][j].x, ray[r].self_k, t_min, bt[r], bk[r]);
                    if (nd[r][j].y < 0.0f) rz_consider(k + 2 * j + 1, nb[r][j].y, nd[r][j].y, ray[r].self_k, t_min, bt[r], bk[r]);
                }
        }
    }
#pragma unroll 1
    for (; k < n_pad; k += 2 * G2, f += 4 * G2) {
        float4 A[G2], B[G2], VA[G2], VB[G2];
#pragma unroll
        for (int j = 0; j < G2; j++) { A[j] = src[f + 4 * j]; B[j] = src[f + 4 * j + 1]; VA[j] = src[f + 4 * j + 2]; VB[j] = src[f + 4 * j + 3]; }
        float2 nb[R][G2], nd[R][G2];
        float m = 1.0f;
#pragma unroll
        for (int r = 0; r < R; r++) {
#pragma unroll
            for (int j = 0; j < G2; j++) {
                rz_test2_moving(A[j], B[j], VA[j], VB[j], q[r], nb[r][j], nd[r][j]);
                m = fminf(m, fminf(nd[r][j].x, nd[r][j].y));
            }
        }
        if (m < 0.0f) {
#pragma unroll
            for (int r = 0; r < R; r++)
#pragma unroll
                for (int j = 0; j < G2; j++) {
                    if (nd[r][j].x < 0.0f) rz_consider(k + 2 * j, nb[r][j].x, nd[r][j].x, ray[r].self_k, t_min, bt[r], bk[r]);
                    if (nd[r][j].y < 0.0f) rz_consider(k + 2 * j + 1, nb[r][j].y, nd[r][j].y, ray[r].self_k, t_min, bt[r], bk[r]);
                }
        }
    }
}

// ------------------------------------------------------------------------------ K1 search over a culled list
// The staged kernels search a LIST of spheres (the primary kernel culls the set against the frustum of its 32-pixel tile, the
// sorted-stage kernel takes the list of its rays' sort group).  Here the packed instructions work on the TWO RAYS of a lane
// (the .x/.y halves hold ray 0 / ray 1) against ONE sphere, whose operands enter as broadcast registers: the same 12 (15)
// issue slots per two tests as the pair form above, but the list has single-sphere granularity.  Round 2's first form kept
// sphere PAIRS in the lists (a pair stays if either half does): 44 tests per ray where the per-sphere lists hold 33.
// Each half follows the operation order of rz_sphere_test exactly (IEEE rn, FTZ): bit-identical (t, k) in every search.
//
// The loop over the list is BRANCH-FREE.  A culled list is dense in hits (one ray in ~30 meets a given sphere of it; some lane
// of the warp nearly always does), so a rare-path branch per sphere was entered all the time: 16 % of the sorted-stage
// kernel's samples sat in it and its reconvergence points (round 1, profiles/r01_sorted_stage_kernel_ncu.md).  Now the only
// thing kept per test is the SIGN of nd, shifted into a per-ray mask by one funnel shift (SHF.L.W: mask = mask << 1 | sign);
// after every 32 spheres the lanes walk the set bits of their masks in one loop — most significant first = list order —
// redo the test of that one sphere with the scalar rz_sphere_test (bit-identical per half) and apply the root rule.  The
// loop runs max-over-lanes(candidates) times instead of once per sphere; a -0.0 or NaN sign is weeded out by the redone test.
// s_cr[k] = (cx, cy, cz, -r^2) of set position k; s_vel[k] = velocity, valid for k >= n_static_pad (the moving part).
// The pairs are held as 64-bit registers through inline PTX (mov.b64 / add|mul|fma.rn.ftz.f32x2): written with the float2
// intrinsics, the compiler kept the rays' scalar registers (they are needed again for shading) and rebuilt every pair with
// two MOVs per use, six per sphere.  Here the pairs are the ONLY copy while the search runs — the scalars are re-read from
// their halves afterwards — which also takes fewer registers than round 2's first form (o, -o, d, -d as scalars per ray).
typedef unsigned long long rz_p2;   // (ray 0, ray 1) or a broadcast (s, s)
__device__ __forceinline__ rz_p2 rz_pack(float x, float y) { rz_p2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y)); return r; }
__device__ __forceinline__ void rz_unpack(rz_p2 v, float &x, float &y) { asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v)); }
__device__ __forceinline__ float rz_half(rz_p2 v, int r) { float x, y; rz_unpack(v, x, y); return r ? y : x; }
__device__ __forceinline__ rz_p2 rz_add2(rz_p2 a, rz_p2 b) { rz_p2 r; asm("add.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ rz_p2 rz_mul2(rz_p2 a, rz_p2 b) { rz_p2 r; asm("mul.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ rz_p2 rz_fma2(rz_p2 a, rz_p2 b, rz_p2 c) { rz_p2 r; asm("fma.rn.ftz.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

// sign flip of both halves as two plain neg.f32: ptxas folds them into the operand modifier of the consuming FFMA2 (-R.F32x2);
// written with neg.ftz (what -x compiles to under --use_fast_math) it emits two FADDs instead.  The values negated here are
// results of FTZ arithmetic, never denormal, so the two agree.
__device__ __forceinline__ rz_p2 rz_neg2(rz_p2 v) {
    float x, y, nx, ny;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v));
    asm("neg.f32 %0, %1;" : "=f"(nx) : "f"(x));
    asm("neg.f32 %0, %1;" : "=f"(ny) : "f"(y));
    rz_p2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(nx), "f"(ny));
    return r;
}

// -o, -d, time of the lane's two rays: seven register pairs (+d enters as a negated operand)
struct RzRay2Ops {
    rz_p2 nox, noy, noz, ndx, ndy, ndz, ntime;   // all negated: a pair that merely copies two scalars is rebuilt by MOVs at every use
};
__device__ __forceinline__ RzRay2Ops rz_ray2_ops(const RzRay (&r)[2]) {
    RzRay2Ops q;
    q.nox = rz_pack(-r[0].o.x, -r[1].o.x); q.noy = rz_pack(-r[0].o.y, -r[1].o.y); q.noz = rz_pack(-r[0].o.z, -r[1].o.z);
    q.ndx = rz_pack(-r[0].d.x, -r[1].d.x); q.ndy = rz_pack(-r[0].d.y, -r[1].d.y); q.ndz = rz_pack(-r[0].d.z, -r[1].d.z);
    q.ntime = rz_pack(-r[0].time, -r[1].time);
    return q;
}
// the rays' scalars back from the pairs (o = -(-o), d = -(-d): exact)
__device__ __forceinline__ void rz_ray2_restore(const RzRay2Ops &q, RzRay (&r)[2]) {
    float a, b;
    rz_unpack(q.nox, a, b); r[0].o.x = -a; r[1].o.x = -b;
    rz_unpack(q.noy, a, b); r[0].o.y = -a; r[1].o.y = -b;
    rz_unpack(q.noz, a, b); r[0].o.z = -a; r[1].o.z = -b;
    rz_unpack(q.ndx, a, b); r[0].d.x = -a; r[1].d.x = -b;
    rz_unpack(q.ndy, a, b); r[0].d.y = -a; r[1].d.y = -b;
    rz_unpack(q.ndz, a, b); r[0].d.z = -a; r[1].d.z = -b;
    rz_unpack(q.ntime, a, b); r[0].time = -a; r[1].time = -b;
}

// sign bits of nd for the two rays against one sphere: the operation order of rz_sphere_test per half
template <bool MOVING>
__device__ __forceinline__ rz_p2 rz_test_r2(const float4 S, const float4 V, const RzRay2Ops &q) {
    rz_p2 ocx = rz_add2(rz_pack(S.x, S.x), q.nox), ocy = rz_add2(rz_pack(S.y, S.y), q.noy), ocz = rz_add2(rz_pack(S.z, S.z), q.noz);
    if (MOVING) {
        ocx = rz_fma2(rz_neg2(rz_pack(V.x, V.x)), q.ntime, ocx);   // v t = (-v)(-t)
        ocy = rz_fma2(rz_neg2(rz_pack(V.y, V.y)), q.ntime, ocy);
        ocz = rz_fma2(rz_neg2(rz_pack(V.z, V.z)), q.ntime, ocz);
    }
    const rz_p2 nb = rz_fma2(ocz, q.ndz, rz_fma2(ocy, q.ndy, rz_mul2(ocx, q.ndx)));
    const rz_p2 b = rz_neg2(nb);                                                               // l = oc + nb d = oc + (-nb)(-d)
    const rz_p2 lx = rz_fma2(b, q.ndx, ocx), ly = rz_fma2(b, q.ndy, ocy), lz = rz_fma2(b, q.ndz, ocz);
    return rz_fma2(lz, lz, rz_fma2(ly, ly, rz_fma2(lx, lx, rz_pack(S.w, S.w))));
}

template <bool MOVING>
__device__ __forceinline__ void rz_resolve_masks(const float4 *__restrict__ s_cr, const float4 *__restrict__ s_vel,
                                                 const unsigned short *__restrict__ list, int cn, unsigned (&m)[2], const RzRay2Ops &q,
                                                 const int (&self_k)[2], float t_min, float (&bt)[2], int (&bk)[2]) {
    unsigned any = m[0] | m[1];
    while (any) {
        any = 0;
#pragma unroll
        for (int r = 0; r < 2; r++) {
            if (m[r]) {
                const int bit = 31 - __clz((int)m[r]);
                m[r] &= ~(1u << bit);
                const int k = list[cn - 1 - bit];           // test number within the chunk
                if (k != (self_k[r] ^ RZ_SELF_OUT)) {       // not the sphere the ray has just left outward (one candidate of ~3 per ray)
                    const float4 S = s_cr[k];
                    float4 V = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (MOVING) V = s_vel[k];
                    float nb, nd;
                    rz_sphere_test(S.x, S.y, S.z, V.x, V.y, V.z, S.w, -rz_half(q.nox, r), -rz_half(q.noy, r), -rz_half(q.noz, r), -rz_half(q.ndx, r),
                                   -rz_half(q.ndy, r), -rz_half(q.ndz, r), -rz_half(q.ntime, r), nb, nd);
                    if (nd < 0.0f) rz_consider(k, nb, nd, self_k[r], t_min, bt[r], bk[r]);
                }
            }
            any |= m[r];
        }
    }
}

template <bool MOVING>
__device__ __forceinline__ void rz_search_list_r2(const float4 *__restrict__ s_cr, const float4 *__restrict__ s_vel,
                                                  const unsigned short *__restrict__ list, int n, const RzRay2Ops &q, const int (&self_k)[2],
                                                  float t_min, float (&bt)[2], int (&bk)[2]) {
#pragma unroll 1
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int cn = min(32, n - i0);
        unsigned m[2] = {0u, 0u};
#pragma unroll 4
        for (int i = 0; i < cn; i++) {
            const int k = list[i0 + i];
            const float4 S = s_cr[k];
            float4 V = make_float4(0.f, 0.f, 0.f, 0.f);
            if (MOVING) V = s_vel[k];
            float n0, n1;
            rz_unpack(rz_test_r2<MOVING>(S, V, q), n0, n1);
            m[0] = __funnelshift_l(__float_as_uint(n0), m[0], 1);
            m[1] = __funnelshift_l(__float_as_uint(n1), m[1], 1);
        }
        rz_resolve_masks<MOVING>(s_cr, s_vel, list + i0, cn, m, q, self_k, t_min, bt, bk);
    }
}

// ls / lm: set positions of the stationary / moving spheres to test, in search order.  The rays' o, d and time live in the
// packed pairs for the duration of the search and are written back from them at the end.
__device__ __forceinline__ void rz_search_lists_r2(const float4 *__restrict__ s_cr, const float4 *__restrict__ s_vel,
                                                   const unsigned short *__restrict__ ls, int n_ls, const unsigned short *__restrict__ lm, int n_lm,
                                                   RzRay (&ray)[2], float t_min, float (&bt)[2], int (&bk)[2]) {
    const RzRay2Ops q = rz_ray2_ops(ray);
    const int self_k[2] = {ray[0].self_k, ray[1].self_k};
    rz_search_list_r2<false>(s_cr, s_vel, ls, n_ls, q, self_k, t_min, bt, bk);
    rz_search_list_r2<true>(s_cr, s_vel, lm, n_lm, q, self_k, t_min, bt, bk);
    rz_ray2_restore(q, ray);
}

// ------------------------------------------------------------------------------ stage scene
// Stage the pair-interleaved sphere set global -> shared with the bulk async-copy engine (cp.async.bulk + mbarrier
// complete_tx; SASS UBLKCP).  All threads of the CTA must call.
__device__ __forceinline__ void rz_stage_scene_pk(const RzSphereSet &set, float4 *s_pk, uint64_t *bar) {
    const uint32_t bytes = (set.n_static_pad + 2u * (set.n_pad - set.n_static_pad)) * 16u;
    if (threadIdx.x == 0) rz_mbar_init(bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        rz_mbar_expect_tx(bar, bytes);
        rz_bulk_g2s(s_pk, set.pk, bytes, bar);
    }
    rz_mbar_wait(bar, 0);
}

// The staged kernels' layout: s_cr[n_pad] = (cx, cy, cz, -r^2) by set position, then the velocities of the moving part
// (s_cr + n_pad; returns the pointer biased so that s_vel[k] is the velocity of set position k >= n_static_pad).
__device__ __forceinline__ const float4 *rz_stage_scene_cv(const RzSphereSet &set, float4 *s_cr, uint64_t *bar) {
    const uint32_t bytes_cr = set.n_pad * 16u, bytes_vel = (set.n_pad - set.n_static_pad) * 16u;
    if (threadIdx.x == 0) rz_mbar_init(bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        rz_mbar_expect_tx(bar, bytes_cr + bytes_vel);
        rz_bulk_g2s(s_cr, set.cr, bytes_cr, bar);
        if (bytes_vel) rz_bulk_g2s(s_cr + set.n_pad, set.vel + set.n_static_pad, bytes_vel, bar);
    }
    rz_mbar_wait(bar, 0);
    return s_cr + set.n_pad - set.n_static_pad;
}

// ------------------------------------------------------------------------------ shade
// Every path kernel has a SOBOL template parameter (RZ_RENDER_SOBOL, RZ_RENDER_RQMC): the launchers pick the instance from
// RzPathArgs::sobol.
// A runtime branch on the field instead raised the registers or spills of the Philox instances (DESIGN.md "Low-discrepancy
// sampling"), which are the default and the benchmark.
// SOBOL = 0 is Philox, 1 Sobol, 2 Sobol with RZ_RENDER_RQMC's replicates and sums: a third instance, because the RQMC code read
// as a uniform bit inside the Sobol instances cost plain Sobol 2 to 4 % of its Mpaths/s.
template <class K>
static inline K rz_pick_sampler(const RzPathArgs &a, K philox, K sobol, K rqmc) {
    return (a.sobol & RZ_SAMPLER_RQMC) ? rqmc : (a.sobol & RZ_SAMPLER_SOBOL) ? sobol : philox;
}

// The instance a launcher runs for (collect_stats, a.sobol).  `inst` names the kernel's instances once, as a
// generic lambda of (std::integral_constant<bool, STATS>, std::integral_constant<int, SOBOL>, std::integral_constant<bool, PASSES>),
// e.g.
//   [](auto S, auto M, auto P) { return rz_second_kernel<decltype(S)::value, decltype(M)::value, decltype(P)::value>; }
// PASSES (RZ_RENDER_PASSES) is an instance of its own for the reason SOBOL is: the default instances carry no trace of it.
template <int V> using rz_int_c = std::integral_constant<int, V>;
template <class F, class S, class P>
static inline auto rz_pick_sampler_of(const RzPathArgs &a, F inst, S stats, P passes) {
    return rz_pick_sampler(a, inst(stats, rz_int_c<0>(), passes), inst(stats, rz_int_c<1>(), passes), inst(stats, rz_int_c<2>(), passes));
}
template <class F>
static inline auto rz_pick_instance(const RzPathArgs &a, int collect_stats, F inst) {
    const std::true_type T{};
    const std::false_type N{};
    if (a.sobol & RZ_PATH_PASSES) return collect_stats ? rz_pick_sampler_of(a, inst, T, T) : rz_pick_sampler_of(a, inst, N, T);
    return collect_stats ? rz_pick_sampler_of(a, inst, T, N) : rz_pick_sampler_of(a, inst, N, N);
}
// The same for a kernel that generates camera rays: `inst` takes a fourth argument, std::integral_constant<bool, FILTER>, and
// FILTER (a pixel filter other than the box in a.sobol, RZ_RENDER_FILTER) is an instance of its own for the same reason.
template <class F>
static inline auto rz_pick_camera_instance(const RzPathArgs &a, int collect_stats, F inst) {
    if (rz_filter_kind(a.sobol) != RZ_FILTER_BOX)
        return rz_pick_instance(a, collect_stats, [inst](auto S, auto M, auto P) { return inst(S, M, P, std::true_type{}); });
    return rz_pick_instance(a, collect_stats, [inst](auto S, auto M, auto P) { return inst(S, M, P, std::false_type{}); });
}

// Grid of a persistent kernel: as many 128-thread CTAs as fit on every SM with `smem` bytes of dynamic shared memory.  The
// attribute that admits that much is set only when smem > 0 (the BVH kernels take none).
template <class K>
static inline cudaError_t rz_persistent_grid(K kern, size_t smem, int sm_count, int *grid) {
    cudaError_t e;
    if (smem > 0 && (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 128, smem)) != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    *grid = sm_count * per_sm;
    return cudaSuccess;
}

enum { RZ_CONT = 0, RZ_END_SKY = 1, RZ_END_ABSORBED = 2, RZ_END_DEPTH = 3 };

// One step of bounceRay (renderer.zig:103-126) after the closest-hit query: miss -> sky and
// accumulate; hit -> refine in f64, scatter, attenuate.  `kind_out` = material kind of the hit.  `sobol`: the kernel's SOBOL
// template argument (0 Philox, 1 RZ_RENDER_SOBOL, 2 with RZ_RENDER_RQMC), a compile-time constant, so that the Philox instances
// carry no trace of the other sampler.  `passes`: the kernel's PASSES template argument (RZ_RENDER_PASSES), likewise: seg also
// carries the first hit's kind (rz_seg_after_hit) and a sky path adds its radiance to its pass too.
__device__ __forceinline__ int rz_shade_segment(const RzPathArgs &a, RzRay &ray, float3 &thr, uint32_t &seg, uint32_t lp,
                                                uint32_t gpix, uint32_t sample, int bk, uint32_t &kind_out, int sobol,
                                                bool passes = false) {
    kind_out = 3u;
    if (bk < 0) {
        // miss: background (renderer.zig:124-125), path ends
        const float3 L = thr * rz_sky(ray.d);
        unsigned long long *acc = a.accum + (size_t)lp * 4u;
        atomicAdd(acc + 0, __float2ull_rn(fminf(fmaxf(L.x, 0.f), 1048576.f) * 4294967296.f));
        atomicAdd(acc + 1, __float2ull_rn(fminf(fmaxf(L.y, 0.f), 1048576.f) * 4294967296.f));
        atomicAdd(acc + 2, __float2ull_rn(fminf(fmaxf(L.z, 0.f), 1048576.f) * 4294967296.f));
        // the noise estimate's second moment (the only accumulation site besides the three above: every kernel shades here)
        if (a.moments) atomicAdd(acc + 3, rz_fixed32(rz_luma_sq(rz_clamp_radiance(L.x), rz_clamp_radiance(L.y), rz_clamp_radiance(L.z))));
        // RZ_RENDER_RQMC: the replicate's luminance sum (rz_pixel_err_rqmc)
        if (sobol == 2)
            atomicAdd(a.accum + rz_rep_offset(a.n_local_px) + (size_t)lp * 2u + (sample & 1u),
                      rz_fixed32(rz_clamp_radiance(rz_luma(rz_clamp_radiance(L.x), rz_clamp_radiance(L.y), rz_clamp_radiance(L.z)))));
        // RZ_RENDER_PASSES: the same three values into the path's pass (the beauty above is never derived from the passes)
        if (passes) {
            unsigned long long *ps = a.accum + rz_pass_offset(a.n_local_px, sobol == 2) +
                                     ((size_t)lp * RZ_PASS_COUNT + rz_pass_of(rz_seg_hits(seg), rz_seg_first_kind(seg))) * 3u;
            atomicAdd(ps + 0, __float2ull_rn(fminf(fmaxf(L.x, 0.f), 1048576.f) * 4294967296.f));
            atomicAdd(ps + 1, __float2ull_rn(fminf(fmaxf(L.y, 0.f), 1048576.f) * 4294967296.f));
            atomicAdd(ps + 2, __float2ull_rn(fminf(fmaxf(L.z, 0.f), 1048576.f) * 4294967296.f));
        }
        return RZ_END_SKY;
    }
    const int k = bk & ~RZ_FAR_BIT;
    const RzHit h = rz_refine_hit(a.set, ray, k, (bk & RZ_FAR_BIT) != 0);
    const uint32_t mat = a.set.mat[k];
    const float4 *mr = a.mats.rec + 4u * mat;
    const float4 m0 = __ldg(mr), m1 = __ldg(mr + 1), m2 = __ldg(mr + 2), m3 = __ldg(mr + 3);
    const uint32_t mbits = __float_as_uint(m0.x);
    RzMatRec M;
    M.kind = mbits & 3u; M.method = (mbits >> 2) & 3u; M.solid = ((mbits >> 4) & 1u) != 0u; M.checker2 = ((mbits >> 5) & 1u) != 0u;
    M.fuzz = m0.y; M.ior = m0.z; M.tex = __float_as_uint(m0.w);
    M.color = f3(m1.x, m1.y, m1.z); M.odd = f3(m2.x, m2.y, m2.z);
    M.inv_scale = __hiloint2double(__float_as_int(m3.y), __float_as_int(m3.x));
    const uint32_t kind = M.kind;
    kind_out = kind < 3u ? kind : 0u;
    if (passes) seg = rz_seg_after_hit(seg, kind_out);
    else seg++;
    const uint32_t hits = passes ? rz_seg_hits(seg) : seg;   // the bounce number every draw and the depth test read
    const uint4 rb = rz_philox(gpix, sample, hits, 0u, a.seed_lo, a.seed_hi);
    const float2 q = sobol ? rz_sobol_u01(a.seed_lo, a.seed_hi, gpix, rz_pair_bounce(hits), sample, sobol == 2)   // u.z, u.w stay Philox
                           : make_float2(rz_u01(rb.x >> 8), rz_u01(rb.y >> 8));
    const float4 u = make_float4(q.x, q.y, rz_u01(rb.z >> 8), rz_u01(rb.w >> 8));
    float3 att;
    if (!rz_scatter(M, a.texs, h, k, u, ray, att)) return RZ_END_ABSORBED;  // black (renderer.zig:109,120)
    thr = thr * att;
    if (hits >= a.max_depth) return RZ_END_DEPTH;  // depth == 0 => black (renderer.zig:104-105)
    return RZ_CONT;
}

// ------------------------------------------------------------------------------ queue helpers
// (the sort key and its decoder, rz_sort_key / rz_key_bounds, live in rz_device.cuh: host + device, property-tested on the CPU)
// Ballot-compacted append of the warp's surviving paths (one atomic per warp).
__device__ __forceinline__ void rz_queue_push(const RzPathArgs &a, bool cont, unsigned lane, unsigned lt_mask, const RzRay &ray, float3 thr,
                                              uint32_t seg, uint32_t lp, uint32_t gpix, uint32_t sample) {
    const unsigned m = __ballot_sync(0xffffffffu, cont);
    if (!m) return;
    unsigned base = 0;
    if (lane == 0) base = atomicAdd(a.q_out_count, (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    const unsigned e = base + __popc(m & lt_mask);
    if (cont && e >= a.queue_cap) atomicOr(a.err, (unsigned)RZ_DEV_ERR_QUEUE_OVERFLOW);   // never silently: the render fails
    if (cont && e < a.queue_cap) {
        float4 *q = a.q_out + (size_t)e * 4u;
        __stcs(q + 0, make_float4(ray.o.x, ray.o.y, ray.o.z, ray.time));
        __stcs(q + 1, make_float4(ray.d.x, ray.d.y, ray.d.z, __int_as_float(ray.self_k)));
        __stcs(q + 2, make_float4(thr.x, thr.y, thr.z, __uint_as_float(seg)));
        __stcs(q + 3, make_float4(__uint_as_float(lp), __uint_as_float(gpix), __uint_as_float(sample), 0.f));
        if (a.q_out_keys) a.q_out_keys[e] = (unsigned short)rz_sort_key(a, ray);
    }
}

// Two rays per lane in one go: one atomic for both ballots (the atomic's round trip, exposed through the shuffle that
// follows it, was ~5 % of the sorted-stage kernel's samples when issued once per ray).
__device__ __forceinline__ void rz_queue_push2(const RzPathArgs &a, const bool (&cont)[2], unsigned lane, unsigned lt_mask, const RzRay (&ray)[2],
                                               const float3 (&thr)[2], const uint32_t (&seg)[2], const uint32_t (&lp)[2], const uint32_t (&gpix)[2],
                                               const uint32_t (&sample)[2]) {
    const unsigned m0 = __ballot_sync(0xffffffffu, cont[0]), m1 = __ballot_sync(0xffffffffu, cont[1]);
    const unsigned n0 = (unsigned)__popc(m0), n1 = (unsigned)__popc(m1);
    if (n0 + n1 == 0u) return;
    unsigned base = 0;
    if (lane == 0) base = atomicAdd(a.q_out_count, n0 + n1);
    base = __shfl_sync(0xffffffffu, base, 0);
    const unsigned e2[2] = {base + (unsigned)__popc(m0 & lt_mask), base + n0 + (unsigned)__popc(m1 & lt_mask)};
#pragma unroll
    for (int r = 0; r < 2; r++) {
        if (cont[r] && e2[r] >= a.queue_cap) atomicOr(a.err, (unsigned)RZ_DEV_ERR_QUEUE_OVERFLOW);
        if (cont[r] && e2[r] < a.queue_cap) {
            float4 *q = a.q_out + (size_t)e2[r] * 4u;
            __stcs(q + 0, make_float4(ray[r].o.x, ray[r].o.y, ray[r].o.z, ray[r].time));
            __stcs(q + 1, make_float4(ray[r].d.x, ray[r].d.y, ray[r].d.z, __int_as_float(ray[r].self_k)));
            __stcs(q + 2, make_float4(thr[r].x, thr[r].y, thr[r].z, __uint_as_float(seg[r])));
            __stcs(q + 3, make_float4(__uint_as_float(lp[r]), __uint_as_float(gpix[r]), __uint_as_float(sample[r]), 0.f));
            if (a.q_out_keys) a.q_out_keys[e2[r]] = (unsigned short)rz_sort_key(a, ray[r]);
        }
    }
}
