// hostsim.cu — TEST INFRASTRUCTURE ONLY (never linked into librayz_cuda.so).
//
// Compiles the product's FP32 device shading code (rayz_b200/csrc/rz_device.cuh: Philox, camera
// ray, f64 hit refinement, scatter, sky, texture) as HOST code and drives it with a scalar
// restatement of the kernel's search/shade loop (rz_path.cu), so the FP32 algorithm's statistics
// can be compared with the f64 oracle in a container without a GPU.  The GPU tests compare the
// real kernels with the oracle; this only de-risks them.
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>
#include <atomic>
#include <algorithm>

#include "../../include/rayz_cuda.h"
#include "../../rayz_b200/csrc/rz_device.cuh"
#include "../../rayz_b200/csrc/rz_host_bvh.hpp"   // the host tree builders (K3's binned-SAH tree): hostsim_bvh_block_check

// the sphere test and the root rule are the product's own (rz_sphere_test / rz_consider, rz_device.cuh)
static inline void consider(int k, float nb, float nd, int self_k, float t_min, float &bt, int &bk) { rz_consider(k, nb, nd, self_k, t_min, bt, bk); }

extern "C" int hostsim_render(const RzScene *sc, const RzCamera *cam, uint32_t w, uint32_t h, uint32_t spp, uint32_t max_depth,
                              uint64_t seed, float t_min, uint32_t threads, double *out_rgb, uint64_t *counters) {
    const uint32_t n = sc->n_spheres;
    std::vector<float4> cr(n), vel(n);
    std::vector<double4> c64(n), v64(n);
    std::vector<uint32_t> smat(n);
    std::vector<int32_t> orig(n);
    for (uint32_t i = 0; i < n; i++) {
        const double *c = sc->sphere_center + 3 * i, *v = sc->sphere_velocity + 3 * i; const double r = sc->sphere_radius[i];
        cr[i] = make_float4((float)c[0], (float)c[1], (float)c[2], -(float)(r * r));
        vel[i] = make_float4((float)v[0], (float)v[1], (float)v[2], (float)r);
        c64[i] = make_double4(c[0], c[1], c[2], r); v64[i] = make_double4(v[0], v[1], v[2], 1.0 / r);
        smat[i] = sc->sphere_material[i]; orig[i] = (int32_t)i;
    }
    const uint32_t nm = sc->n_materials, nt = sc->n_textures;
    std::vector<uint32_t> mk(nm), mt(nm), mm(nm), tk(nt), te(nt), to(nt);
    std::vector<float> mf(nm), mi(nm); std::vector<float4> tc(nt); std::vector<double> ts(nt);
    for (uint32_t i = 0; i < nm; i++) { mk[i] = sc->mat_kind[i]; mt[i] = sc->mat_kind[i] == 2 ? 0 : sc->mat_texture[i]; mm[i] = sc->mat_method ? sc->mat_method[i] : 2; mf[i] = (float)sc->mat_fuzz[i]; mi[i] = (float)sc->mat_ior[i]; }
    for (uint32_t i = 0; i < nt; i++) { tk[i] = sc->tex_kind[i]; te[i] = sc->tex_even[i]; to[i] = sc->tex_odd[i];
        tc[i] = make_float4((float)sc->tex_color[3*i], (float)sc->tex_color[3*i+1], (float)sc->tex_color[3*i+2], 0); ts[i] = sc->tex_kind[i] == 0 ? 1.0 / sc->tex_scale[i] : 0; }
    RzSphereSet S; S.cr = cr.data(); S.vel = vel.data(); S.c64 = c64.data(); S.v64 = v64.data(); S.mat = smat.data(); S.orig = orig.data(); S.n = n; S.n_static = 0; S.n_static_pad = 0; S.n_pad = n;
    RzMaterials M; M.kind = mk.data(); M.fuzz = mf.data(); M.ior = mi.data(); M.tex = mt.data(); M.method = mm.data();
    RzTextures T; T.kind = tk.data(); T.color = tc.data(); T.inv_scale = ts.data(); T.even = te.data(); T.odd = to.data();
    RzCamF32 C;
    C.look_from = make_float3((float)cam->look_from[0], (float)cam->look_from[1], (float)cam->look_from[2]);
    C.px_du = make_float3((float)cam->px_du[0], (float)cam->px_du[1], (float)cam->px_du[2]);
    C.px_dv = make_float3((float)cam->px_dv[0], (float)cam->px_dv[1], (float)cam->px_dv[2]);
    C.px_origin = make_float3((float)cam->px_origin[0], (float)cam->px_origin[1], (float)cam->px_origin[2]);
    C.defocus_u = make_float3((float)cam->defocus_u[0], (float)cam->defocus_u[1], (float)cam->defocus_u[2]);
    C.defocus_v = make_float3((float)cam->defocus_v[0], (float)cam->defocus_v[1], (float)cam->defocus_v[2]);
    C.defocus = cam->defocus;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    if (!(t_min > 0)) t_min = 1e-4f;
    if (threads == 0) threads = std::max(1u, std::thread::hardware_concurrency());
    std::atomic<uint32_t> next(0);
    std::vector<std::vector<uint64_t>> cnt(threads, std::vector<uint64_t>(10, 0));
    auto work = [&](uint32_t tid) {
        uint64_t *ct = cnt[tid].data();
        while (true) {
            const uint32_t j = next.fetch_add(1);
            if (j >= h) break;
            for (uint32_t i = 0; i < w; i++) {
                unsigned long long acc[3] = {0, 0, 0};
                const uint32_t gpix = j * w + i;
                for (uint32_t s = 0; s < spp; s++) {
                    RzRay ray = rz_camera_ray(C, i, j, gpix, s, k0, k1);
                    float3 thr = f3(1, 1, 1);
                    uint32_t seg = 0;
                    bool alive = max_depth > 0;
                    ct[0]++;
                    if (!alive) ct[9]++;
                    while (alive) {
                        float bt = 3.0e38f; int bk = -1;
                        for (uint32_t k = 0; k < n; k++) {
                            const float4 sp = cr[k], v = vel[k];
                            float nb, nd;
                            rz_sphere_test(sp.x, sp.y, sp.z, v.x, v.y, v.z, sp.w, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, ray.time, nb, nd);
                            if (nd < 0.0f) consider((int)k, nb, nd, ray.self_k, t_min, bt, bk);
                        }
                        ct[1]++;
                        if (bk < 0) {
                            const float3 L = thr * rz_sky(ray.d);
                            acc[0] += (unsigned long long)llrintf(fminf(fmaxf(L.x, 0.f), 1048576.f) * 4294967296.f);
                            acc[1] += (unsigned long long)llrintf(fminf(fmaxf(L.y, 0.f), 1048576.f) * 4294967296.f);
                            acc[2] += (unsigned long long)llrintf(fminf(fmaxf(L.z, 0.f), 1048576.f) * 4294967296.f);
                            ct[7]++;
                            break;
                        }
                        const int k = bk & ~RZ_FAR_BIT;
                        const RzHit hit = rz_refine_hit(S, ray, k, (bk & RZ_FAR_BIT) != 0);
                        const uint32_t mat = S.mat[k], kind = M.kind[mat];
                        ct[4 + kind]++;
                        seg++;
                        const uint4 rb = rz_philox(gpix, s, seg, 0u, k0, k1);
                        const float4 u = make_float4(rz_u01(rb.x >> 8), rz_u01(rb.y >> 8), rz_u01(rb.z >> 8), rz_u01(rb.w >> 8));
                        float3 att;
                        // decoded from the SoA arrays, and always through the texture walk: an independent check of the
                        // flattened per-material records (and their solid-colour shortcut) the device kernels read
                        RzMatRec R;
                        R.kind = kind; R.method = M.method[mat]; R.tex = M.tex[mat]; R.solid = false; R.checker2 = false;
                        R.fuzz = M.fuzz[mat]; R.ior = M.ior[mat]; R.color = f3(0.f, 0.f, 0.f);
                        if (!rz_scatter(R, T, hit, k, u, ray, att)) { ct[8]++; break; }
                        thr = thr * att;
                        if (seg >= max_depth) { ct[9]++; break; }
                    }
                }
                const double inv = 1.0 / (double)spp, sc32 = 2.3283064365386962890625e-10;
                for (int c = 0; c < 3; c++) out_rgb[((size_t)j * w + i) * 3 + c] = (double)acc[c] * sc32 * inv;
            }
        }
    };
    std::vector<std::thread> pool;
    for (uint32_t t = 0; t < threads; t++) pool.emplace_back(work, t);
    for (auto &t : pool) t.join();
    if (counters) { for (int i = 0; i < 10; i++) { counters[i] = 0; for (auto &c : cnt) counters[i] += c[i]; } counters[2] = counters[1] * n; }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Path by path, for the f64 replay (oracle Scene.replay, tests/test_replay_cpu.py): the paths of samples [sample_offset,
// sample_offset + spp) of every pixel, pixel-major, each through the product's camera, sphere test, root rule, refinement,
// scatter and sky, with the uniforms rz_shade_segment draws (rz_search.cuh:397-401) for sampler 0 (Philox), 1 (Sobol) or
// 2 (Sobol-RQMC), and the material records as the library packs them (solid and checker-of-two-solids shortcuts,
// rz_context.cu).  Outputs per path: rgb[3] clamped f32 radiance, segs, end (0 sky, 1 absorbed, 2 depth), hits[3].
// ---------------------------------------------------------------------------------------------
extern "C" int hostsim_paths(const RzScene *sc, const RzCamera *cam, uint32_t w, uint32_t h, uint32_t sample_offset, uint32_t spp,
                             uint32_t max_depth, uint64_t seed, float t_min, int sampler, uint32_t threads, float *out_rgb,
                             uint32_t *out_segs, uint8_t *out_end, uint32_t *out_hits) {
    const uint32_t n = sc->n_spheres;
    std::vector<float4> cr(n), vel(n);
    std::vector<double4> c64(n), v64(n);
    std::vector<uint32_t> smat(n);
    std::vector<int32_t> orig(n);
    for (uint32_t i = 0; i < n; i++) {
        const double *c = sc->sphere_center + 3 * i, *v = sc->sphere_velocity + 3 * i; const double r = sc->sphere_radius[i];
        cr[i] = make_float4((float)c[0], (float)c[1], (float)c[2], -(float)(r * r));
        vel[i] = make_float4((float)v[0], (float)v[1], (float)v[2], (float)r);
        c64[i] = make_double4(c[0], c[1], c[2], r); v64[i] = make_double4(v[0], v[1], v[2], 1.0 / r);
        smat[i] = sc->sphere_material[i]; orig[i] = (int32_t)i;
    }
    const uint32_t nm = sc->n_materials, nt = sc->n_textures;
    std::vector<uint32_t> tk(nt), te(nt), to(nt);
    std::vector<float4> tc(nt); std::vector<double> ts(nt);
    for (uint32_t i = 0; i < nt; i++) { tk[i] = sc->tex_kind[i]; te[i] = sc->tex_even[i]; to[i] = sc->tex_odd[i];
        tc[i] = make_float4((float)sc->tex_color[3*i], (float)sc->tex_color[3*i+1], (float)sc->tex_color[3*i+2], 0); ts[i] = sc->tex_kind[i] == 0 ? 1.0 / sc->tex_scale[i] : 0; }
    std::vector<RzMatRec> recs(nm);
    for (uint32_t i = 0; i < nm; i++) {
        RzMatRec &R = recs[i];
        R.kind = sc->mat_kind[i]; R.method = sc->mat_method ? sc->mat_method[i] : 2u; R.tex = R.kind == 2u ? 0u : sc->mat_texture[i];
        R.fuzz = (float)sc->mat_fuzz[i]; R.ior = (float)sc->mat_ior[i];
        const bool textured = R.kind != 2u && nt > 0;
        R.solid = textured && tk[R.tex] != 0u;
        R.checker2 = textured && !R.solid && tk[te[R.tex]] != 0u && tk[to[R.tex]] != 0u;
        const float4 even = R.solid ? tc[R.tex] : R.checker2 ? tc[te[R.tex]] : make_float4(0, 0, 0, 0), odd = R.checker2 ? tc[to[R.tex]] : make_float4(0, 0, 0, 0);
        R.color = f3(even.x, even.y, even.z); R.odd = f3(odd.x, odd.y, odd.z);
        R.inv_scale = R.checker2 ? ts[R.tex] : 0.0;
    }
    RzSphereSet S; S.cr = cr.data(); S.vel = vel.data(); S.c64 = c64.data(); S.v64 = v64.data(); S.mat = smat.data(); S.orig = orig.data(); S.n = n; S.n_static = 0; S.n_static_pad = 0; S.n_pad = n;
    RzTextures T; T.kind = tk.data(); T.color = tc.data(); T.inv_scale = ts.data(); T.even = te.data(); T.odd = to.data();
    RzCamF32 C;
    C.look_from = make_float3((float)cam->look_from[0], (float)cam->look_from[1], (float)cam->look_from[2]);
    C.px_du = make_float3((float)cam->px_du[0], (float)cam->px_du[1], (float)cam->px_du[2]);
    C.px_dv = make_float3((float)cam->px_dv[0], (float)cam->px_dv[1], (float)cam->px_dv[2]);
    C.px_origin = make_float3((float)cam->px_origin[0], (float)cam->px_origin[1], (float)cam->px_origin[2]);
    C.defocus_u = make_float3((float)cam->defocus_u[0], (float)cam->defocus_u[1], (float)cam->defocus_u[2]);
    C.defocus_v = make_float3((float)cam->defocus_v[0], (float)cam->defocus_v[1], (float)cam->defocus_v[2]);
    C.defocus = cam->defocus;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    if (!(t_min > 0)) t_min = 1e-4f;
    if (threads == 0) threads = std::max(1u, std::thread::hardware_concurrency());
    std::atomic<uint32_t> next(0);
    auto work = [&]() {
        while (true) {
            const uint32_t j = next.fetch_add(1);
            if (j >= h) break;
            for (uint32_t i = 0; i < w; i++) {
                const uint32_t gpix = j * w + i;
                for (uint32_t sl = 0; sl < spp; sl++) {
                    const size_t q = (size_t)gpix * spp + sl;
                    const uint32_t sample = sample_offset + sl;
                    RzRay ray = rz_camera_ray(C, i, j, gpix, sample, k0, k1, sampler);
                    float3 thr = f3(1, 1, 1), L = f3(0, 0, 0);
                    uint32_t seg = 0, segs = 0, hits[3] = {0, 0, 0};
                    uint8_t end = 2;
                    bool alive = max_depth > 0;
                    while (alive) {
                        float bt = 3.0e38f; int bk = -1;
                        for (uint32_t k = 0; k < n; k++) {
                            float nb, nd;
                            rz_sphere_test(cr[k].x, cr[k].y, cr[k].z, vel[k].x, vel[k].y, vel[k].z, cr[k].w, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, ray.time, nb, nd);
                            if (nd < 0.0f) consider((int)k, nb, nd, ray.self_k, t_min, bt, bk);
                        }
                        segs++;
                        if (bk < 0) {   // rz_shade_segment's miss branch
                            const float3 c = thr * rz_sky(ray.d);
                            L = f3(rz_clamp_radiance(c.x), rz_clamp_radiance(c.y), rz_clamp_radiance(c.z));
                            end = 0;
                            break;
                        }
                        const int k = bk & ~RZ_FAR_BIT;
                        const RzHit hit = rz_refine_hit(S, ray, k, (bk & RZ_FAR_BIT) != 0);
                        const RzMatRec &M = recs[smat[k]];
                        hits[M.kind < 3u ? M.kind : 0u]++;
                        seg++;
                        const uint4 rb = rz_philox(gpix, sample, seg, 0u, k0, k1);
                        const float2 qq = sampler ? rz_sobol_u01(k0, k1, gpix, rz_pair_bounce(seg), sample, sampler == 2)
                                                  : make_float2(rz_u01(rb.x >> 8), rz_u01(rb.y >> 8));
                        const float4 u = make_float4(qq.x, qq.y, rz_u01(rb.z >> 8), rz_u01(rb.w >> 8));
                        float3 att;
                        if (!rz_scatter(M, T, hit, k, u, ray, att)) { end = 1; break; }
                        thr = thr * att;
                        if (seg >= max_depth) break;
                    }
                    out_rgb[3 * q] = L.x; out_rgb[3 * q + 1] = L.y; out_rgb[3 * q + 2] = L.z;
                    out_segs[q] = segs; out_end[q] = end;
                    for (int c = 0; c < 3; c++) out_hits[3 * q + c] = hits[c];
                }
            }
        }
    };
    std::vector<std::thread> pool;
    for (uint32_t t = 0; t < threads; t++) pool.emplace_back(work);
    for (auto &t : pool) t.join();
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Property check of the staged K1's sort key (rz_device.cuh: rz_key_grid / rz_sort_key / rz_key_bounds): for random rays
// in and around the sphere box, the bounds decoded from a ray's key must contain the ray — origin inside the key's cell
// box, direction signs equal to the key's octant, exit time from the sphere box below the key's reach bound.  The
// sorted-stage kernel culls spheres from exactly these bounds, so a violation here would be a missed hit there.
// Returns the number of violations; counts[0..15] = rays per reach class, counts[16] = distinct keys seen.
// ---------------------------------------------------------------------------------------------
// direction field of the sort key in the checks below: -1 = chosen by the shape of the box (the product's default), 0 = octants, 1 = sectors
static int g_key_mode = -1;
extern "C" void hostsim_set_key_mode(int m) { g_key_mode = m; }
static double g_huge_factor = 4.0;   // experiment knob: spheres above this multiple of the median radius stay outside the sphere box
extern "C" void hostsim_set_huge_factor(double f) { g_huge_factor = f; }
static int g_cell_bits = 9;
extern "C" void hostsim_set_cell_bits(int b) { g_cell_bits = b; }

extern "C" uint64_t hostsim_key_check(const float *lo, const float *hi, int cell_bits, uint64_t n_rays, uint64_t seed, uint64_t *counts) {
    RzPathArgs a;
    memset(&a, 0, sizeof a);
    const float l3[3] = {lo[0], lo[1], lo[2]}, h3[3] = {hi[0], hi[1], hi[2]};
    rz_key_grid(a, l3, h3, cell_bits, g_key_mode);
    std::vector<unsigned char> seen(65536, 0);
    uint64_t s = seed * 0x9E3779B97F4A7C15ull + 1, bad = 0;
    auto u01 = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return (float)((s >> 40) * (1.0 / 16777216.0)); };
    for (int i = 0; i < 17; i++) counts[i] = 0;
    for (uint64_t r = 0; r < n_rays; r++) {
        RzRay ray;
        float o[3], d[3];
        for (int ax = 0; ax < 3; ax++) {
            const float e = h3[ax] - l3[ax];
            o[ax] = l3[ax] + e * (1.6f * u01() - 0.3f);            // 30 % of the extent beyond the box on either side
            if (u01() < 0.02f) o[ax] = u01() < 0.5f ? l3[ax] : h3[ax];   // exactly on a face
            d[ax] = 2.0f * u01() - 1.0f;
            if (u01() < 0.03f) d[ax] = u01() < 0.5f ? 0.0f : -0.0f;     // axis-parallel rays
            if (u01() < 0.03f) d[ax] *= 1e-6f;                          // grazing
        }
        const float len = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
        if (!(len > 1e-12f)) { d[0] = 0.f; d[1] = 1.f; d[2] = 0.f; } else { d[0] /= len; d[1] /= len; d[2] /= len; }
        ray.o = f3(o[0], o[1], o[2]); ray.d = f3(d[0], d[1], d[2]); ray.time = 0.f; ray.self_k = -1;
        const uint32_t key = rz_sort_key(a, ray);
        if (key > 0xffffu) { bad++; continue; }
        float blo[3], bhi[3], T;
        uint32_t oct;
        rz_key_bounds(a, key, blo, bhi, oct, T);
        bool ok = true;
        for (int ax = 0; ax < 3; ax++) {
            ok = ok && o[ax] >= blo[ax] && o[ax] <= bhi[ax];
            if (!a.key_sectors) ok = ok && (((oct >> ax) & 1u) != 0u) == (d[ax] < 0.f);
        }
        if (a.key_sectors) {   // sector of the projection on the (key_u, key_w) plane
            const float du = d[a.key_u], dw = d[a.key_w];
            ok = ok && ((oct & 1u) != 0u) == (du < 0.f) && ((oct & 2u) != 0u) == (dw < 0.f) && ((oct & 4u) != 0u) == (fabsf(du) < fabsf(dw));
            if (a.key_sectors == 2u)   // sixteen sectors: + the half of the 45-degree wedge (next to the axis <=> bit 3)
                ok = ok && ((oct & 8u) != 0u) == (fminf(fabsf(du), fabsf(dw)) < RZ_TAN_22_5 * fmaxf(fabsf(du), fabsf(dw)));
            else ok = ok && oct < 8u;
        }
        {   // the reach the key stands for: the stay inside the sphere box — with sector keys, its projection on the (u, w) plane
            float reach = rz_box_exit(a, ray);
            if (a.key_sectors) reach *= sqrtf(d[a.key_u] * d[a.key_u] + d[a.key_w] * d[a.key_w]);
            ok = ok && reach <= T;
        }
        if (!ok) bad++;
        counts[key & 15u]++;
        if (!seen[key]) { seen[key] = 1; counts[16]++; }
    }
    return bad;
}

// ---------------------------------------------------------------------------------------------
// Property checks of the two culls of the staged K1 (rz_device.cuh: rz_tile_keep, rz_unit_keep): a sphere that one of the
// rays HITS (the kernels' own FP32 test, sphere evaluated at the ray's time) must never be culled.  Spheres are generated
// around points on the rays, so about half of them are hit.  out[0] = violations, out[1] = hits checked, out[2] = hit
// spheres the cull kept (== out[1] when there is no violation), out[3] = misses the cull dropped (it does cull).
// ---------------------------------------------------------------------------------------------
namespace {
struct Rng {
    uint64_t s;
    explicit Rng(uint64_t seed) : s(seed * 0x9E3779B97F4A7C15ull + 0x1234567ull) {}
    float u01() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return (float)((s >> 40) * (1.0 / 16777216.0)); }
    float sym() { return 2.0f * u01() - 1.0f; }
};

// the kernels' sphere test: does the line hit, and is a root ahead of t_min?
bool ray_hits(const RzRay &ray, const float c0[3], const float v[3], float r, float t_min) {
    const float ocx = fmaf(v[0], ray.time, c0[0] - ray.o.x), ocy = fmaf(v[1], ray.time, c0[1] - ray.o.y), ocz = fmaf(v[2], ray.time, c0[2] - ray.o.z);
    const float b = fmaf(ocz, ray.d.z, fmaf(ocy, ray.d.y, ocx * ray.d.x));
    const float c = fmaf(ocz, ocz, fmaf(ocy, ocy, fmaf(ocx, ocx, -(r * r))));
    const float disc = fmaf(b, b, -c);
    return disc > 0.0f && b + sqrtf(disc) > t_min;
}

// a sphere near the point the ray reaches at parameter t: centre at the ray's time within 1.5 r of it
void sphere_near(Rng &g, const RzRay &ray, float t, float r, float vmax, float c0[3], float v[3]) {
    const float p[3] = {ray.o.x + t * ray.d.x, ray.o.y + t * ray.d.y, ray.o.z + t * ray.d.z};
    const bool moving = g.u01() < 0.6f;
    for (int ax = 0; ax < 3; ax++) {
        v[ax] = moving ? vmax * g.sym() : 0.0f;
        c0[ax] = p[ax] + 1.5f * r * g.sym() * 0.8f - v[ax] * ray.time;
    }
}
}  // namespace

extern "C" int hostsim_tile_cull_check(const RzCamera *cam, uint32_t w, uint32_t h, uint64_t n_tiles, uint64_t seed, uint64_t *out) {
    RzCamF32 C;
    C.look_from = make_float3((float)cam->look_from[0], (float)cam->look_from[1], (float)cam->look_from[2]);
    C.px_du = make_float3((float)cam->px_du[0], (float)cam->px_du[1], (float)cam->px_du[2]);
    C.px_dv = make_float3((float)cam->px_dv[0], (float)cam->px_dv[1], (float)cam->px_dv[2]);
    C.px_origin = make_float3((float)cam->px_origin[0], (float)cam->px_origin[1], (float)cam->px_origin[2]);
    C.defocus_u = make_float3((float)cam->defocus_u[0], (float)cam->defocus_u[1], (float)cam->defocus_u[2]);
    C.defocus_v = make_float3((float)cam->defocus_v[0], (float)cam->defocus_v[1], (float)cam->defocus_v[2]);
    C.defocus = cam->defocus;
    // the two thin-lens numbers the library derives from the camera (rz_context.cu, enqueue_staged)
    double pcd[3], lu = 0, lv = 0, f2 = 0;
    for (int ax = 0; ax < 3; ax++) {
        pcd[ax] = cam->px_origin[ax] + 0.5 * (w - 1) * cam->px_du[ax] + 0.5 * (h - 1) * cam->px_dv[ax] - cam->look_from[ax];
        f2 += pcd[ax] * pcd[ax]; lu += cam->defocus_u[ax] * cam->defocus_u[ax]; lv += cam->defocus_v[ax] * cam->defocus_v[ax];
    }
    const float focus_dist = (float)std::sqrt(f2);
    const float lens_radius = cam->defocus ? (float)(std::sqrt(std::max(lu, lv)) * 1.001) : 0.f;
    Rng g(seed);
    for (int i = 0; i < 4; i++) out[i] = 0;
    const uint32_t n_px = w * h;
    for (uint64_t t = 0; t < n_tiles; t++) {
        const uint32_t tile = (uint32_t)(g.u01() * (float)((n_px + 31u) / 32u)) % ((n_px + 31u) / 32u);
        // ---- the cone, lane by lane as the kernel builds it
        float3 ax = f3(0.f, 0.f, 0.f), pcs[32];
        uint32_t pis[32], pjs[32];
        bool valid[32];
        for (uint32_t lane = 0; lane < 32; lane++) {
            const uint32_t lp = tile * 32u + lane;
            valid[lane] = lp < n_px;
            pis[lane] = pjs[lane] = 0;
            if (valid[lane]) rz_local_to_global(lp, w, 0, 1, 4, pis[lane], pjs[lane]);
            pcs[lane] = rz_tile_pixel_dir(C, pis[lane], pjs[lane]);
            if (valid[lane]) ax = ax + normalize3(pcs[lane]);
        }
        const bool has_axis = rz_tile_axis(ax);
        float cmin = 1.0f;
        for (uint32_t lane = 0; lane < 32; lane++)
            if (valid[lane]) cmin = fminf(cmin, rz_tile_corner_cos(C, pcs[lane], ax));
        const RzTileCone cone = rz_tile_cone(C, ax, has_axis, cmin, focus_dist, lens_radius);
        // ---- camera rays of the tile against spheres placed around them
        for (int k = 0; k < 64; k++) {
            const uint32_t lane = (uint32_t)(g.u01() * 32.f) & 31u;
            if (!valid[lane]) continue;
            const uint32_t gpix = pjs[lane] * w + pis[lane], sample = (uint32_t)(g.u01() * 4096.f);
            const RzRay ray = rz_camera_ray(C, pis[lane], pjs[lane], gpix, sample, (uint32_t)seed, 77u);
            for (int j = 0; j < 6; j++) {
                const float tt = 0.05f + 40.0f * g.u01() * g.u01();
                const float r = 0.03f + 2.0f * g.u01() * g.u01();
                float c0[3], v[3];
                sphere_near(g, ray, tt, r, j < 2 ? 6.0f : 0.8f, c0, v);
                const bool hit = ray_hits(ray, c0, v, r, 1e-4f);
                const bool kept = rz_tile_keep(cone, c0[0], c0[1], c0[2], v[0], v[1], v[2], -(r * r));
                if (hit) { out[1]++; if (kept) out[2]++; else out[0]++; }
                else if (!kept) out[3]++;
            }
        }
    }
    return 0;
}

// K3's camera stage (rz_bvh_stage_kernel with tile lists): work units are 8 x 4 pixel blocks and the TREE is culled against the
// block's cone — a box as its bounding sphere (rz_tile_keep_box).  For camera rays of random blocks and spheres placed around
// them: a sphere a ray hits must be kept, and so must every box that contains the sphere's sweep over the shutter — its own
// FP32 box and ever larger ancestors (grown by random amounts on every side, up to thousands of units).
// out: [0] hit spheres dropped, [1] hits, [2] boxes around hit spheres dropped, [3] boxes tested, [4] misses culled
extern "C" int hostsim_block_cull_check(const RzCamera *cam, uint32_t w, uint32_t h, uint64_t n_blocks, uint64_t seed, uint64_t *out) {
    RzCamF32 C;
    C.look_from = make_float3((float)cam->look_from[0], (float)cam->look_from[1], (float)cam->look_from[2]);
    C.px_du = make_float3((float)cam->px_du[0], (float)cam->px_du[1], (float)cam->px_du[2]);
    C.px_dv = make_float3((float)cam->px_dv[0], (float)cam->px_dv[1], (float)cam->px_dv[2]);
    C.px_origin = make_float3((float)cam->px_origin[0], (float)cam->px_origin[1], (float)cam->px_origin[2]);
    C.defocus_u = make_float3((float)cam->defocus_u[0], (float)cam->defocus_u[1], (float)cam->defocus_u[2]);
    C.defocus_v = make_float3((float)cam->defocus_v[0], (float)cam->defocus_v[1], (float)cam->defocus_v[2]);
    C.defocus = cam->defocus;
    double pcd[3], lu = 0, lv = 0, f2 = 0;
    for (int ax = 0; ax < 3; ax++) {
        pcd[ax] = cam->px_origin[ax] + 0.5 * (w - 1) * cam->px_du[ax] + 0.5 * (h - 1) * cam->px_dv[ax] - cam->look_from[ax];
        f2 += pcd[ax] * pcd[ax]; lu += cam->defocus_u[ax] * cam->defocus_u[ax]; lv += cam->defocus_v[ax] * cam->defocus_v[ax];
    }
    const float focus_dist = (float)std::sqrt(f2);
    const float lens_radius = cam->defocus ? (float)(std::sqrt(std::max(lu, lv)) * 1.001) : 0.f;
    Rng g(seed);
    for (int i = 0; i < 5; i++) out[i] = 0;
    const uint32_t tiles_x = (w + 7u) / 8u, tiles_y = (h + 3u) / 4u, n_px = w * h;
    for (uint64_t t = 0; t < n_blocks; t++) {
        const uint32_t tile = (uint32_t)(g.u01() * (float)(tiles_x * tiles_y)) % (tiles_x * tiles_y);
        // ---- the block's pixels as the kernel maps them (RzPathArgs::tile_w = 8), then the cone, lane by lane
        float3 ax = f3(0.f, 0.f, 0.f), pcs[32];
        uint32_t pis[32], pjs[32];
        bool valid[32];
        const uint32_t ty = tile / tiles_x, tx = tile - ty * tiles_x;
        for (uint32_t lane = 0; lane < 32; lane++) {
            const uint32_t ti = tx * 8u + (lane & 7u), tr = ty * 4u + (lane >> 3);
            const uint32_t lp = tr * w + ti;
            valid[lane] = ti < w && lp < n_px;
            pis[lane] = pjs[lane] = 0;
            if (valid[lane]) rz_local_to_global(lp, w, 0, 1, 4, pis[lane], pjs[lane]);
            pcs[lane] = rz_tile_pixel_dir(C, pis[lane], pjs[lane]);
            if (valid[lane]) ax = ax + normalize3(pcs[lane]);
        }
        const bool has_axis = rz_tile_axis(ax);
        float cmin = 1.0f;
        for (uint32_t lane = 0; lane < 32; lane++)
            if (valid[lane]) cmin = fminf(cmin, rz_tile_corner_cos(C, pcs[lane], ax));
        const RzTileCone cone = rz_tile_cone(C, ax, has_axis, cmin, focus_dist, lens_radius);
        for (int k = 0; k < 64; k++) {
            const uint32_t lane = (uint32_t)(g.u01() * 32.f) & 31u;
            if (!valid[lane]) continue;
            const uint32_t gpix = pjs[lane] * w + pis[lane], sample = (uint32_t)(g.u01() * 4096.f);
            const RzRay ray = rz_camera_ray(C, pis[lane], pjs[lane], gpix, sample, (uint32_t)seed, 77u);
            for (int j = 0; j < 6; j++) {
                const float tt = 0.05f + (j == 5 ? 400.0f : 40.0f) * g.u01() * g.u01();       // some far away: config 4's rays travel hundreds of units
                const float r = j == 4 ? 1000.0f : 0.03f + 2.0f * g.u01() * g.u01();          // and a ground-sized sphere
                float c0[3], v[3];
                sphere_near(g, ray, tt, r, j < 2 ? 6.0f : 0.8f, c0, v);
                const bool hit = ray_hits(ray, c0, v, r, 1e-4f);
                const bool kept = rz_tile_keep(cone, c0[0], c0[1], c0[2], v[0], v[1], v[2], -(r * r));
                if (!hit) { if (!kept) out[4]++; continue; }
                out[1]++;
                if (!kept) out[0]++;
                // the sphere's box over the shutter (Sphere.boundingBox), rounded outward, then ever larger enclosing boxes
                float lo[3], hi[3];
                for (int a3 = 0; a3 < 3; a3++) {
                    const float a0 = c0[a3], a1 = c0[a3] + v[a3];
                    lo[a3] = nextafterf(fminf(a0, a1) - r, -INFINITY);
                    hi[a3] = nextafterf(fmaxf(a0, a1) + r, INFINITY);
                }
                float grow = 0.0f;
                for (int level = 0; level < 8; level++) {
                    out[3]++;
                    if (!rz_tile_keep_box(cone, lo[0], hi[0], lo[1], hi[1], lo[2], hi[2])) out[2]++;
                    grow = level == 0 ? 0.05f : grow * 5.0f;                                   // 0.05 ... 3900 units
                    for (int a3 = 0; a3 < 3; a3++) { lo[a3] -= grow * g.u01(); hi[a3] += grow * g.u01(); }
                }
            }
        }
    }
    return 0;
}

extern "C" int hostsim_unit_cull_check(const float *lo, const float *hi, int cell_bits, float huge_radius, uint64_t n_units, uint64_t seed,
                                       uint64_t *out) {
    RzPathArgs a;
    memset(&a, 0, sizeof a);
    const float l3[3] = {lo[0], lo[1], lo[2]}, h3[3] = {hi[0], hi[1], hi[2]};
    rz_key_grid(a, l3, h3, cell_bits, g_key_mode);
    a.huge_radius = huge_radius;
    Rng g(seed);
    for (int i = 0; i < 4; i++) out[i] = 0;
    const float ext = std::max(h3[0] - l3[0], std::max(h3[1] - l3[1], h3[2] - l3[2]));
    for (uint64_t u = 0; u < n_units; u++) {
        // ---- a unit: rays that start close together and head roughly the same way (what the sort puts side by side)
        RzRay rays[16];
        float bo[3], bd[3];
        for (int ax = 0; ax < 3; ax++) { bo[ax] = l3[ax] + (h3[ax] - l3[ax]) * (1.3f * g.u01() - 0.15f); bd[ax] = g.sym(); }
        const float spread = g.u01() < 0.5f ? 0.05f : 0.6f, jitter = ext / 64.0f * g.u01();
        RzUnitBounds U;
        rz_unit_bounds_init(U);
        int cls[16];
        for (int k = 0; k < 16; k++) {
            float d[3];
            for (int ax = 0; ax < 3; ax++) d[ax] = bd[ax] + spread * g.sym();
            const float len = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
            if (!(len > 1e-6f)) { d[0] = 0.f; d[1] = 1.f; d[2] = 0.f; } else { d[0] /= len; d[1] /= len; d[2] /= len; }
            rays[k].o = f3(bo[0] + jitter * g.sym(), bo[1] + jitter * g.sym(), bo[2] + jitter * g.sym());
            rays[k].d = f3(d[0], d[1], d[2]); rays[k].time = g.u01(); rays[k].self_k = -1;
            const uint32_t key = rz_sort_key(a, rays[k]);
            rz_unit_bounds_add_cell(U, a, key);     // the unit's box and common signs come from the cells and octants ...
            cls[k] = (int)(key & 15u);              // ... each ray keeps its own reach class
        }
        // ---- spheres around the rays: ordinary ones lie inside the sphere box over the whole shutter interval (that is
        // what the box is), huge ones anywhere
        for (int k = 0; k < 16; k++) {
            for (int j = 0; j < 8; j++) {
                const bool huge = j == 7;
                const float r = huge ? huge_radius * (1.5f + 50.f * g.u01()) : fminf(huge_radius, 0.02f * ext * (0.1f + g.u01()));
                // j == 6: a sphere BEHIND the ray's origin (never hit; a coherent unit's sign test should drop it)
                const float tt = j == 6 ? -(0.05f * ext + 0.5f * ext * g.u01()) : 0.02f * ext + 1.2f * ext * g.u01() * g.u01();
                float c0[3], v[3];
                sphere_near(g, rays[k], tt, r, j < 3 ? 0.1f * ext : 0.01f * ext, c0, v);
                bool inside = true;
                for (int ax = 0; ax < 3 && !huge; ax++) {
                    const float p0 = c0[ax], p1 = c0[ax] + v[ax];
                    inside = inside && fminf(p0, p1) - r >= l3[ax] && fmaxf(p0, p1) + r <= h3[ax];
                }
                if (!inside) continue;
                const bool hit = ray_hits(rays[k], c0, v, r, 1e-4f);
                // the sorted-stage kernel gives a ray of reach class c the spheres of classes <= c (rz_unit_class)
                const bool kept = rz_unit_class(U, a, c0[0], c0[1], c0[2], v[0], v[1], v[2], -(r * r)) <= cls[k];
                if (hit) { out[1]++; if (kept) out[2]++; else out[0]++; }
                else if (!kept) out[3]++;
            }
        }
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// The staged K1 on a real scene, stage by stage, on the CPU: camera rays searched over their tile's culled list, scattered
// rays grouped by sort key and searched over their group's culled list — each against the brute-force
// search over every sphere.  The closest hit (t and sphere) must be identical, which is the claim the staged form rests on
// ("the culls only ever drop spheres a ray cannot reach").  Uses the functions the kernels call (rz_device.cuh).
// out[0] = mismatches (primary), out[1] = primary rays, out[2] = sum of primary list sizes,
// out[3] = mismatches (sorted units), out[4] = rays in units, out[5] = sum of list sizes (per ray), out[6] = groups.
// ---------------------------------------------------------------------------------------------
extern "C" int hostsim_staged_check(const RzScene *sc, const RzCamera *cam, uint32_t w, uint32_t h, uint32_t spp, uint32_t tile_stride,
                                    uint64_t seed, uint64_t *out) {
    const uint32_t n = sc->n_spheres;
    std::vector<float4> cr(n), vel(n);
    std::vector<double4> c64(n), v64(n);
    std::vector<uint32_t> smat(n);
    std::vector<int32_t> orig(n);
    for (uint32_t i = 0; i < n; i++) {
        const double *c = sc->sphere_center + 3 * i, *v = sc->sphere_velocity + 3 * i; const double r = sc->sphere_radius[i];
        cr[i] = make_float4((float)c[0], (float)c[1], (float)c[2], -(float)(r * r));
        vel[i] = make_float4((float)v[0], (float)v[1], (float)v[2], (float)r);
        c64[i] = make_double4(c[0], c[1], c[2], r); v64[i] = make_double4(v[0], v[1], v[2], 1.0 / r);
        smat[i] = sc->sphere_material[i]; orig[i] = (int32_t)i;
    }
    const uint32_t nm = sc->n_materials, nt = sc->n_textures;
    std::vector<uint32_t> mk(nm), mt(nm), mm(nm), tk(nt), te(nt), to(nt);
    std::vector<float> mf(nm), mi(nm); std::vector<float4> tc(nt); std::vector<double> ts(nt);
    for (uint32_t i = 0; i < nm; i++) { mk[i] = sc->mat_kind[i]; mt[i] = sc->mat_kind[i] == 2 ? 0 : sc->mat_texture[i]; mm[i] = sc->mat_method ? sc->mat_method[i] : 2; mf[i] = (float)sc->mat_fuzz[i]; mi[i] = (float)sc->mat_ior[i]; }
    for (uint32_t i = 0; i < nt; i++) { tk[i] = sc->tex_kind[i]; te[i] = sc->tex_even[i]; to[i] = sc->tex_odd[i];
        tc[i] = make_float4((float)sc->tex_color[3*i], (float)sc->tex_color[3*i+1], (float)sc->tex_color[3*i+2], 0); ts[i] = sc->tex_kind[i] == 0 ? 1.0 / sc->tex_scale[i] : 0; }
    RzSphereSet S; S.cr = cr.data(); S.vel = vel.data(); S.c64 = c64.data(); S.v64 = v64.data(); S.mat = smat.data(); S.orig = orig.data(); S.n = n; S.n_static = 0; S.n_static_pad = 0; S.n_pad = n;
    RzTextures T; T.kind = tk.data(); T.color = tc.data(); T.inv_scale = ts.data(); T.even = te.data(); T.odd = to.data();
    RzCamF32 C;
    C.look_from = make_float3((float)cam->look_from[0], (float)cam->look_from[1], (float)cam->look_from[2]);
    C.px_du = make_float3((float)cam->px_du[0], (float)cam->px_du[1], (float)cam->px_du[2]);
    C.px_dv = make_float3((float)cam->px_dv[0], (float)cam->px_dv[1], (float)cam->px_dv[2]);
    C.px_origin = make_float3((float)cam->px_origin[0], (float)cam->px_origin[1], (float)cam->px_origin[2]);
    C.defocus_u = make_float3((float)cam->defocus_u[0], (float)cam->defocus_u[1], (float)cam->defocus_u[2]);
    C.defocus_v = make_float3((float)cam->defocus_v[0], (float)cam->defocus_v[1], (float)cam->defocus_v[2]);
    C.defocus = cam->defocus;
    double f2 = 0, lu = 0, lv = 0;
    for (int ax = 0; ax < 3; ax++) {
        const double pc = cam->px_origin[ax] + 0.5 * (w - 1) * cam->px_du[ax] + 0.5 * (h - 1) * cam->px_dv[ax] - cam->look_from[ax];
        f2 += pc * pc; lu += cam->defocus_u[ax] * cam->defocus_u[ax]; lv += cam->defocus_v[ax] * cam->defocus_v[ax];
    }
    const float focus_dist = (float)std::sqrt(f2), lens_radius = cam->defocus ? (float)(std::sqrt(std::max(lu, lv)) * 1.001) : 0.f;
    // the sphere box as the library sets it up at upload (rz_context.cu: box of the spheres rz_huge_threshold leaves inside,
    // motion over the shutter included, padded by 0.1 % + 1e-3)
    RzPathArgs a;
    memset(&a, 0, sizeof a);
    {
        const double huge = rz_huge_threshold(sc->sphere_radius, n, g_huge_factor);
        double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
        bool any = false;
        for (uint32_t i = 0; i < n; i++) {
            if (sc->sphere_radius[i] > huge) continue;
            any = true;
            for (int ax = 0; ax < 3; ax++) {
                const double c0 = sc->sphere_center[3 * i + ax], c1 = c0 + sc->sphere_velocity[3 * i + ax], r = sc->sphere_radius[i];
                lo[ax] = std::min(lo[ax], std::min(c0, c1) - r); hi[ax] = std::max(hi[ax], std::max(c0, c1) + r);
            }
        }
        float l3[3], h3[3];
        for (int ax = 0; ax < 3; ax++) {
            const double pad = any ? 1e-3 * (hi[ax] - lo[ax]) + 1e-3 : 0.0;
            l3[ax] = any ? (float)(lo[ax] - pad) : -3.0e38f; h3[ax] = any ? (float)(hi[ax] + pad) : 3.0e38f;
        }
        rz_key_grid(a, l3, h3, g_cell_bits, g_key_mode);
        a.huge_radius = (float)huge;
    }
    const float t_min = 1e-4f;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int i = 0; i < 7; i++) out[i] = 0;
    auto search = [&](const RzRay &ray, const std::vector<uint32_t> *list, float &bt, int &bk) {
        bt = 3.0e38f; bk = -1;
        const uint32_t cnt = list ? (uint32_t)list->size() : n;
        for (uint32_t q = 0; q < cnt; q++) {
            const uint32_t k = list ? (*list)[q] : q;
            const float4 sp = cr[k], v = vel[k];
            float nb, nd;
            rz_sphere_test(sp.x, sp.y, sp.z, v.x, v.y, v.z, sp.w, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, ray.time, nb, nd);
            if (nd < 0.0f) consider((int)k, nb, nd, ray.self_k, t_min, bt, bk);
        }
    };
    struct Entry { uint32_t key; RzRay ray; };
    std::vector<Entry> queue;
    const uint32_t n_px = w * h, n_tiles = (n_px + 31u) / 32u;
    std::vector<uint32_t> list;
    for (uint32_t tile = 0; tile < n_tiles; tile += std::max(1u, tile_stride)) {
        // ---- primary kernel: the tile's cone and list
        float3 ax = f3(0.f, 0.f, 0.f), pcs[32];
        uint32_t pis[32], pjs[32];
        bool valid[32];
        for (uint32_t lane = 0; lane < 32; lane++) {
            const uint32_t lp = tile * 32u + lane;
            valid[lane] = lp < n_px;
            pis[lane] = pjs[lane] = 0;
            if (valid[lane]) rz_local_to_global(lp, w, 0, 1, 4, pis[lane], pjs[lane]);
            pcs[lane] = rz_tile_pixel_dir(C, pis[lane], pjs[lane]);
            if (valid[lane]) ax = ax + normalize3(pcs[lane]);
        }
        const bool has_axis = rz_tile_axis(ax);
        float cmin = 1.0f;
        for (uint32_t lane = 0; lane < 32; lane++)
            if (valid[lane]) cmin = fminf(cmin, rz_tile_corner_cos(C, pcs[lane], ax));
        const RzTileCone cone = rz_tile_cone(C, ax, has_axis, cmin, focus_dist, lens_radius);
        list.clear();
        for (uint32_t k = 0; k < n; k++)
            if (rz_tile_keep(cone, cr[k].x, cr[k].y, cr[k].z, vel[k].x, vel[k].y, vel[k].z, cr[k].w)) list.push_back(k);
        for (uint32_t lane = 0; lane < 32; lane++) {
            if (!valid[lane]) continue;
            const uint32_t gpix = pjs[lane] * w + pis[lane];
            for (uint32_t s = 0; s < spp; s++) {
                RzRay ray = rz_camera_ray(C, pis[lane], pjs[lane], gpix, s, k0, k1);
                float bt, bt2; int bk, bk2;
                search(ray, nullptr, bt, bk);
                search(ray, &list, bt2, bk2);
                out[1]++; out[2] += list.size();
                if (bk != bk2 || bt != bt2) out[0]++;
                if (bk < 0) continue;
                // scatter, as rz_shade_segment does, and queue the new ray under its key
                const int k = bk & ~RZ_FAR_BIT;
                const RzHit hit = rz_refine_hit(S, ray, k, (bk & RZ_FAR_BIT) != 0);
                const uint32_t mat = smat[k];
                RzMatRec R;
                R.kind = mk[mat]; R.method = mm[mat]; R.tex = mt[mat]; R.solid = false; R.checker2 = false; R.fuzz = mf[mat]; R.ior = mi[mat]; R.color = f3(0.f, 0.f, 0.f);
                const uint4 rb = rz_philox(gpix, s, 1u, 0u, k0, k1);
                const float4 u = make_float4(rz_u01(rb.x >> 8), rz_u01(rb.y >> 8), rz_u01(rb.z >> 8), rz_u01(rb.w >> 8));
                float3 att;
                if (!rz_scatter(R, T, hit, k, u, ray, att)) continue;
                queue.push_back(Entry{rz_sort_key(a, ray), ray});
            }
        }
    }
    // ---- sorted-stage kernel: entries grouped by (cell, direction field) = key >> 4 (rz_sort.cu); a work unit never straddles
    // two groups, so every ray searches its group's pair list (rz_bin_lists_kernel: every sphere's smallest reach class from
    // the group's own cell and direction, rz_unit_class) up to its own class c: the spheres of classes <= c
    std::stable_sort(queue.begin(), queue.end(), [](const Entry &x, const Entry &y) { return (x.key >> 4) < (y.key >> 4); });
    std::vector<int> scls(n);
    for (size_t e0 = 0; e0 < queue.size();) {
        size_t e1 = e0;
        while (e1 < queue.size() && (queue[e1].key >> 4) == (queue[e0].key >> 4)) e1++;
        RzUnitBounds U;
        rz_unit_bounds_init(U);
        rz_unit_bounds_add_cell(U, a, queue[e0].key);
        for (uint32_t k = 0; k < n; k++) scls[k] = rz_unit_class(U, a, cr[k].x, cr[k].y, cr[k].z, vel[k].x, vel[k].y, vel[k].z, cr[k].w);
        out[6]++;
        for (size_t i = e0; i < e1; i++) {
            const int c = (int)(queue[i].key & 15u);
            list.clear();
            for (uint32_t k = 0; k < n; k++) if (scls[k] <= c) list.push_back(k);
            float bt, bt2; int bk, bk2;
            search(queue[i].ray, nullptr, bt, bk);
            search(queue[i].ray, &list, bt2, bk2);
            out[4]++; out[5] += list.size();
            if (getenv("HS_DBG")) { static uint64_t hr[16], hl[16]; hr[c]++; hl[c] += list.size(); if (i + 1 == queue.size()) for (int q = 0; q < 16; q++) fprintf(stderr, "class %d rays %llu avg list %.1f T %.2f\n", q, (unsigned long long)hr[q], hr[q] ? (double)hl[q] / hr[q] : 0.0, rz_class_T(a, q)); }
            if (bk != bk2 || bt != bt2) out[3]++;
        }
        e0 = e1;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// K3's camera stage on a real scene, on the CPU: the library's own binned-SAH tree (rz_host_bvh.hpp) is culled against the cone
// of every `block_stride`-th 8 x 4 pixel block exactly as rz_bvh_stage_kernel does it (breadth first from the root, a child box
// through rz_tile_keep_box, a leaf's spheres through rz_tile_keep), and `spp` camera rays per pixel of the block are searched
// over the surviving spheres and over EVERY sphere with the kernels' sphere test and root rule: the closest hit (t and sphere)
// must be the same.  out[0] = rays whose hit differs, out[1] = rays, out[2] = sum of list sizes over the blocks, out[3] = blocks,
// out[4] = blocks whose list would outgrow `cap` (the kernel walks the tree per ray there), out[5] = largest frontier.
// ---------------------------------------------------------------------------------------------
extern "C" int hostsim_bvh_block_check(const RzScene *sc, const RzCamera *cam, uint32_t w, uint32_t h, uint32_t spp, uint32_t block_stride,
                                       uint32_t cap, uint64_t seed, uint64_t *out) {
    const uint32_t n = sc->n_spheres;
    SahBuilder sb;
    sb.p.resize(n);
    for (uint32_t i = 0; i < n; i++) {
        sb.p[i].b = sphere_box(*sc, i);
        for (int a = 0; a < 3; a++) sb.p[i].c[a] = 0.5 * (sb.p[i].b.lo[a] + sb.p[i].b.hi[a]);
        sb.p[i].s = i;
    }
    sb.run();
    // the set in leaf order, as the library uploads it
    std::vector<float4> cr(n), vel(n);
    for (uint32_t k = 0; k < n; k++) {
        const uint32_t i = sb.order[k];
        const double *c = sc->sphere_center + 3 * i, *v = sc->sphere_velocity + 3 * i; const double r = sc->sphere_radius[i];
        cr[k] = make_float4((float)c[0], (float)c[1], (float)c[2], -(float)(r * r));
        vel[k] = make_float4((float)v[0], (float)v[1], (float)v[2], (float)r);
    }
    RzCamF32 C;
    C.look_from = make_float3((float)cam->look_from[0], (float)cam->look_from[1], (float)cam->look_from[2]);
    C.px_du = make_float3((float)cam->px_du[0], (float)cam->px_du[1], (float)cam->px_du[2]);
    C.px_dv = make_float3((float)cam->px_dv[0], (float)cam->px_dv[1], (float)cam->px_dv[2]);
    C.px_origin = make_float3((float)cam->px_origin[0], (float)cam->px_origin[1], (float)cam->px_origin[2]);
    C.defocus_u = make_float3((float)cam->defocus_u[0], (float)cam->defocus_u[1], (float)cam->defocus_u[2]);
    C.defocus_v = make_float3((float)cam->defocus_v[0], (float)cam->defocus_v[1], (float)cam->defocus_v[2]);
    C.defocus = cam->defocus;
    double f2 = 0, lu = 0, lv = 0;
    for (int ax = 0; ax < 3; ax++) {
        const double pc = cam->px_origin[ax] + 0.5 * (w - 1) * cam->px_du[ax] + 0.5 * (h - 1) * cam->px_dv[ax] - cam->look_from[ax];
        f2 += pc * pc; lu += cam->defocus_u[ax] * cam->defocus_u[ax]; lv += cam->defocus_v[ax] * cam->defocus_v[ax];
    }
    const float focus_dist = (float)std::sqrt(f2), lens_radius = cam->defocus ? (float)(std::sqrt(std::max(lu, lv)) * 1.001) : 0.f;
    for (int i = 0; i < 6; i++) out[i] = 0;
    const uint32_t tiles_x = (w + 7u) / 8u, tiles_y = (h + 3u) / 4u, n_px = w * h;
    std::vector<int> frontier, next, list;
    for (uint32_t tile = 0; tile < tiles_x * tiles_y; tile += block_stride) {
        float3 ax = f3(0.f, 0.f, 0.f), pcs[32];
        uint32_t pis[32], pjs[32];
        bool valid[32];
        const uint32_t ty = tile / tiles_x, tx = tile - ty * tiles_x;
        for (uint32_t lane = 0; lane < 32; lane++) {
            const uint32_t ti = tx * 8u + (lane & 7u), tr = ty * 4u + (lane >> 3);
            const uint32_t lp = tr * w + ti;
            valid[lane] = ti < w && lp < n_px;
            pis[lane] = pjs[lane] = 0;
            if (valid[lane]) rz_local_to_global(lp, w, 0, 1, 4, pis[lane], pjs[lane]);
            pcs[lane] = rz_tile_pixel_dir(C, pis[lane], pjs[lane]);
            if (valid[lane]) ax = ax + normalize3(pcs[lane]);
        }
        const bool has_axis = rz_tile_axis(ax);
        float cmin = 1.0f;
        for (uint32_t lane = 0; lane < 32; lane++)
            if (valid[lane]) cmin = fminf(cmin, rz_tile_corner_cos(C, pcs[lane], ax));
        const RzTileCone cone = rz_tile_cone(C, ax, has_axis, cmin, focus_dist, lens_radius);
        // ---- the cull: breadth first from the root
        frontier.assign(1, 0);
        list.clear();
        while (!frontier.empty()) {
            out[5] = std::max<uint64_t>(out[5], frontier.size());
            next.clear();
            for (int node : frontier) {
                const RzBvhNode &nd = sb.nodes[(size_t)node];
                for (int c = 0; c < 2; c++) {
                    if (nd.child[c] < 0 && nd.cnt[c] == 0u) continue;      // unused slot (the library fills it with the sibling: same spheres)
                    if (!rz_tile_keep_box(cone, nd.lox[c], nd.hix[c], nd.loy[c], nd.hiy[c], nd.loz[c], nd.hiz[c])) continue;
                    if (nd.child[c] >= 0) { next.push_back(nd.child[c]); continue; }
                    const int first = ~nd.child[c];
                    for (uint32_t e = 0; e < nd.cnt[c]; e++) {
                        const int k = first + (int)e;
                        if (rz_tile_keep(cone, cr[k].x, cr[k].y, cr[k].z, vel[k].x, vel[k].y, vel[k].z, cr[k].w)) list.push_back(k);
                    }
                }
            }
            frontier.swap(next);
        }
        out[2] += list.size(); out[3]++;
        if (list.size() > cap) out[4]++;
        // ---- the block's camera rays: the list against every sphere
        for (uint32_t lane = 0; lane < 32; lane++) {
            if (!valid[lane]) continue;
            const uint32_t gpix = pjs[lane] * w + pis[lane];
            for (uint32_t smp = 0; smp < spp; smp++) {
                const RzRay ray = rz_camera_ray(C, pis[lane], pjs[lane], gpix, smp, (uint32_t)seed, (uint32_t)(seed >> 32));
                float bt_l = 3.0e38f, bt_a = 3.0e38f;
                int bk_l = -1, bk_a = -1;
                for (int k : list) {
                    float nb, nd2;
                    rz_sphere_test(cr[k].x, cr[k].y, cr[k].z, vel[k].x, vel[k].y, vel[k].z, cr[k].w, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, ray.time, nb, nd2);
                    if (nd2 < 0.0f) rz_consider(k, nb, nd2, -1, 1e-4f, bt_l, bk_l);
                }
                for (int k = 0; k < (int)n; k++) {
                    float nb, nd2;
                    rz_sphere_test(cr[k].x, cr[k].y, cr[k].z, vel[k].x, vel[k].y, vel[k].z, cr[k].w, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, ray.time, nb, nd2);
                    if (nd2 < 0.0f) rz_consider(k, nb, nd2, -1, 1e-4f, bt_a, bk_a);
                }
                out[1]++;
                if (bk_l != bk_a || bt_l != bt_a) out[0]++;
            }
        }
    }
    return 0;
}
