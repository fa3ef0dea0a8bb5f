// Test-only: the pixel filters' warp (rz_device.cuh's rz_filter_warp), the Sobol jitter it is fed, and the two camera-stage
// culls with a filter's footprint (rz_tile_corner_cos's half-width) compiled as HOST code, so that tests/test_filter_cpu.py can
// check them on the CPU.  The product only ever runs these functions inside its CUDA kernels.
#include <cmath>
#include <cstdint>
#include <thread>
#include <vector>

#include "../../rayz_b200/csrc/rz_device.cuh"

// out[i] = rz_filter_warp(kind, width16, u[i]), on `threads` threads
extern "C" void hostfilt_warp(uint32_t kind, uint32_t width16, const float *u, uint64_t n, float *out, int threads) {
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; t++)
        pool.emplace_back([=] {
            for (uint64_t i = (uint64_t)t; i < n; i += (uint64_t)threads) out[i] = rz_filter_warp(kind, width16, u[i]);
        });
    for (auto &th : pool) th.join();
}

extern "C" uint32_t hostfilt_width16(uint32_t flags) { return rz_filter_width16(flags); }
extern "C" float hostfilt_reach(uint32_t flags) { return rz_filter_reach(flags); }

// The camera-jitter pair of samples [s0, s0 + n) of pixel gpix under RZ_RENDER_SOBOL (rqmc: RZ_RENDER_RQMC's replicates),
// and the camera ray's image-plane offsets under the filter of `flags`: rz_camera_ray's own arithmetic.
extern "C" void hostfilt_sobol_jitter(uint32_t k0, uint32_t k1, uint32_t gpix, uint32_t s0, uint32_t n, int rqmc, uint32_t flags,
                                      float *ux, float *uy, float *wx, float *wy) {
    const uint32_t kind = rz_filter_kind(flags), w16 = rz_filter_width16(flags);
    for (uint32_t i = 0; i < n; i++) {
        const float2 j = rz_sobol_u01(k0, k1, gpix, RZ_PAIR_CAMERA_JITTER, s0 + i, rqmc != 0);
        ux[i] = j.x; uy[i] = j.y;
        wx[i] = rz_filter_warp(kind, w16, j.x); wy[i] = rz_filter_warp(kind, w16, j.y);
    }
}

// The camera ray of one sample from explicit uniforms: (o, d) of rz_lens_ray under the filter of `flags`.
extern "C" void hostfilt_lens_ray(const RzCamera *cam, uint32_t px, uint32_t py, const float *u5, uint32_t flags, float *od) {
    RzCamF32 C;
    C.look_from = make_float3((float)cam->look_from[0], (float)cam->look_from[1], (float)cam->look_from[2]);
    C.px_du = make_float3((float)cam->px_du[0], (float)cam->px_du[1], (float)cam->px_du[2]);
    C.px_dv = make_float3((float)cam->px_dv[0], (float)cam->px_dv[1], (float)cam->px_dv[2]);
    C.px_origin = make_float3((float)cam->px_origin[0], (float)cam->px_origin[1], (float)cam->px_origin[2]);
    C.defocus_u = make_float3((float)cam->defocus_u[0], (float)cam->defocus_u[1], (float)cam->defocus_u[2]);
    C.defocus_v = make_float3((float)cam->defocus_v[0], (float)cam->defocus_v[1], (float)cam->defocus_v[2]);
    C.defocus = cam->defocus;
    const RzRay r = rz_lens_ray(C, px, py, u5[0], u5[1], u5[2], u5[3], u5[4], flags & RZ_PATH_FILTER_BITS);
    od[0] = r.o.x; od[1] = r.o.y; od[2] = r.o.z; od[3] = r.d.x; od[4] = r.d.y; od[5] = r.d.z;
}

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

// a sphere near the point the ray reaches at parameter t: centre at the ray's time within 1.2 r of it
void sphere_near(Rng &g, const RzRay &ray, float t, float r, float vmax, float c0[3], float v[3]) {
    const float p[3] = {ray.o.x + t * ray.d.x, ray.o.y + t * ray.d.y, ray.o.z + t * ray.d.z};
    const bool moving = g.u01() < 0.6f;
    for (int ax = 0; ax < 3; ax++) {
        v[ax] = moving ? vmax * g.sym() : 0.0f;
        c0[ax] = p[ax] + 1.5f * r * g.sym() * 0.8f - v[ax] * ray.time;
    }
}

// a jitter uniform: a quarter of them at the ends of the support (u = 0: w = -R; u = 1: w = +R, exactly), the rest uniform
float jitter(Rng &g) {
    const float e = g.u01();
    return e < 0.125f ? 0.0f : e < 0.25f ? 1.0f : g.u01();
}
}  // namespace

// Both camera-stage culls under a pixel filter (`flags`), on the pixel layouts the kernels use: block = 0 is the staged K1's
// 32-pixel tile (rz_primary_kernel, rz_tile_keep), block = 1 K3's 8 x 4 block (rz_bvh_stage_kernel: rz_tile_keep for spheres,
// rz_tile_keep_box for the boxes around them).  The cone is built as the kernels build it, with the corners at
// +-rz_filter_reach(flags) (cone_half > 0: at +-cone_half instead, to show what a narrower cone drops); the rays start at
// filtered offsets, a quarter of them exactly at +-R, from anywhere on the lens.
// out: [0] hit spheres dropped, [1] hits, [2] boxes around hit spheres dropped, [3] boxes tested, [4] misses culled
extern "C" int hostfilt_cull_check(const RzCamera *cam, uint32_t w, uint32_t h, int block, uint32_t flags, float cone_half,
                                   uint64_t n_units, uint64_t seed, uint64_t *out) {
    RzCamF32 C;
    C.look_from = make_float3((float)cam->look_from[0], (float)cam->look_from[1], (float)cam->look_from[2]);
    C.px_du = make_float3((float)cam->px_du[0], (float)cam->px_du[1], (float)cam->px_du[2]);
    C.px_dv = make_float3((float)cam->px_dv[0], (float)cam->px_dv[1], (float)cam->px_dv[2]);
    C.px_origin = make_float3((float)cam->px_origin[0], (float)cam->px_origin[1], (float)cam->px_origin[2]);
    C.defocus_u = make_float3((float)cam->defocus_u[0], (float)cam->defocus_u[1], (float)cam->defocus_u[2]);
    C.defocus_v = make_float3((float)cam->defocus_v[0], (float)cam->defocus_v[1], (float)cam->defocus_v[2]);
    C.defocus = cam->defocus;
    // the two thin-lens numbers the library derives from the camera (rz_context.cu, enqueue_staged)
    double lu = 0, lv = 0, f2 = 0;
    for (int ax = 0; ax < 3; ax++) {
        const double pc = cam->px_origin[ax] + 0.5 * (w - 1) * cam->px_du[ax] + 0.5 * (h - 1) * cam->px_dv[ax] - cam->look_from[ax];
        f2 += pc * pc; lu += cam->defocus_u[ax] * cam->defocus_u[ax]; lv += cam->defocus_v[ax] * cam->defocus_v[ax];
    }
    const float focus_dist = (float)std::sqrt(f2);
    const float lens_radius = cam->defocus ? (float)(std::sqrt(std::max(lu, lv)) * 1.001) : 0.f;
    const uint32_t bits = flags & RZ_PATH_FILTER_BITS;
    const float half = cone_half > 0.f ? cone_half : rz_filter_reach(bits);
    Rng g(seed);
    for (int i = 0; i < 5; i++) out[i] = 0;
    const uint32_t n_px = w * h, tiles_x = (w + 7u) / 8u, n_blocks = tiles_x * ((h + 3u) / 4u), n_tiles = (n_px + 31u) / 32u;
    for (uint64_t t = 0; t < n_units; t++) {
        const uint32_t n = block ? n_blocks : n_tiles;
        const uint32_t tile = (uint32_t)(g.u01() * (float)n) % n;
        float3 ax = f3(0.f, 0.f, 0.f), pcs[32];
        uint32_t pis[32], pjs[32];
        bool valid[32];
        for (uint32_t lane = 0; lane < 32; lane++) {
            uint32_t lp;
            if (block) {
                const uint32_t ty = tile / tiles_x, tx = tile - ty * tiles_x, ti = tx * 8u + (lane & 7u);
                lp = (ty * 4u + (lane >> 3)) * w + ti;
                valid[lane] = ti < w && lp < n_px;
            } else {
                lp = tile * 32u + lane;
                valid[lane] = lp < n_px;
            }
            pis[lane] = pjs[lane] = 0;
            if (valid[lane]) rz_local_to_global(lp, w, 0, 1, 4, pis[lane], pjs[lane]);
            pcs[lane] = rz_tile_pixel_dir(C, pis[lane], pjs[lane]);
            if (valid[lane]) ax = ax + normalize3(pcs[lane]);
        }
        const bool has_axis = rz_tile_axis(ax);
        float cmin = 1.0f;
        for (uint32_t lane = 0; lane < 32; lane++)
            if (valid[lane]) cmin = fminf(cmin, rz_tile_corner_cos(C, pcs[lane], ax, half));
        const RzTileCone cone = rz_tile_cone(C, ax, has_axis, cmin, focus_dist, lens_radius);
        for (int k = 0; k < 64; k++) {
            const uint32_t lane = (uint32_t)(g.u01() * 32.f) & 31u;
            if (!valid[lane]) continue;
            const float ux = jitter(g), uy = jitter(g), ut = g.u01(), ur = g.u01() < 0.25f ? 1.0f : g.u01(), ua = g.u01();
            const RzRay ray = rz_lens_ray(C, pis[lane], pjs[lane], ux, uy, ut, ur, ua, bits);
            for (int j = 0; j < 6; j++) {
                const float tt = 0.05f + (j == 5 ? 400.0f : 40.0f) * g.u01() * g.u01();
                const float r = j == 4 ? 1000.0f : 0.03f + 2.0f * g.u01() * g.u01();
                float c0[3], v[3];
                sphere_near(g, ray, tt, r, j < 2 ? 6.0f : 0.8f, c0, v);
                const bool hit = ray_hits(ray, c0, v, r, 1e-4f);
                const bool kept = rz_tile_keep(cone, c0[0], c0[1], c0[2], v[0], v[1], v[2], -(r * r));
                if (!hit) { if (!kept) out[4]++; continue; }
                out[1]++;
                if (!kept) out[0]++;
                if (!block) continue;
                // the sphere's box over the shutter, rounded outward, then ever larger enclosing boxes
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
                    grow = level == 0 ? 0.05f : grow * 5.0f;
                    for (int a3 = 0; a3 < 3; a3++) { lo[a3] -= grow * g.u01(); hi[a3] += grow * g.u01(); }
                }
            }
        }
    }
    return 0;
}
