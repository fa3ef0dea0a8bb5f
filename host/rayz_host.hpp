// rayz_host.hpp — C++ stand-in for the reference's Zig host code above the C ABI.
//
// The reference is compiled Zig and no zig toolchain exists in this image, so the host side is
// written in C++ with the reference's own type and function names, argument meaning and error
// behaviour (a failed backend call surfaces as an exception where Zig returns an error union):
//
//   V3, Ray                      vec.zig:4-167
//   Camera::init                 camera.zig:18-57
//   MemPool / Handle             ecs.zig:6-70
//   Sphere, Material, Texture    geom.zig:11-22, material.zig:19-51,73-165
//   Image / writePPM             image.zig:4-41
//   Tracer::init / render        renderer.zig:18-101   <- render() is the drop-in seam
//   DefaultPrng / float(f64)     Zig std.Random (xoshiro256++ via SplitMix64)
//   randomBouncing               rayz.zig:45-168
//
// Nothing here traces rays: Tracer::render flattens the pool, calls rayz_cuda_upload_scene +
// rayz_cuda_render and widens the float result back into Image::pixels.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../include/rayz_cuda.h"

namespace rayz {

struct V3 {
    double x = 0, y = 0, z = 0;
    static V3 of(double v) { return {v, v, v}; }
    static V3 ones() { return of(1); }
    static V3 y_hat() { return {0, 1, 0}; }
    V3 add(V3 o) const { return {x + o.x, y + o.y, z + o.z}; }
    V3 sub(V3 o) const { return {x - o.x, y - o.y, z - o.z}; }
    V3 mul(double v) const { return {x * v, y * v, z * v}; }
    V3 div(double v) const { return mul(1 / v); }  // vec.zig:67-69
    double dot(V3 o) const { return x * o.x + y * o.y + z * o.z; }
    double mag() const { return std::sqrt(dot(*this)); }
    V3 unit() const { return div(mag()); }
    V3 cross(V3 o) const { return {y * o.z - z * o.y, z * o.x - x * o.z, x * o.y - y * o.x}; }
    V3 vmul(V3 o) const { return {x * o.x, y * o.y, z * o.z}; }
};

struct Ray {
    V3 origin, dir;
    double time = 0;
};

// std.Random.DefaultPrng + Random.float(f64)
struct DefaultPrng {
    uint64_t s[4];
    explicit DefaultPrng(uint64_t seed) {
        uint64_t sm = seed;
        for (int i = 0; i < 4; i++) {
            sm += 0x9e3779b97f4a7c15ull;
            uint64_t z = sm;
            z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
            z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
            s[i] = z ^ (z >> 31);
        }
    }
    static uint64_t rotl(uint64_t v, int k) { return (v << k) | (v >> (64 - k)); }
    uint64_t next() {
        const uint64_t r = rotl(s[0] + s[3], 23) + s[0];
        const uint64_t t = s[1] << 17;
        s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = rotl(s[3], 45);
        return r;
    }
    double float64() {
        const uint64_t rand = next();
        uint64_t lz = rand ? (uint64_t)__builtin_clzll(rand) : 64;
        if (lz >= 12) {
            lz = 12;
            while (true) {
                const uint64_t v = next();
                const uint64_t addl = v ? (uint64_t)__builtin_clzll(v) : 64;
                lz += addl;
                if (addl != 64) break;
                if (lz >= 1022) { lz = 1022; break; }
            }
        }
        const uint64_t bits = ((1022 - lz) << 52) | (rand & 0xFFFFFFFFFFFFFull);
        double d;
        std::memcpy(&d, &bits, 8);
        return d;
    }
    V3 v3(double low, double high) {  // V3.random, vec.zig:9-16
        const double scale = high - low;
        V3 r;
        r.x = float64() * scale + low;
        r.y = float64() * scale + low;
        r.z = float64() * scale + low;
        return r;
    }
};

struct Camera {
    V3 look_from, px_du, px_dv, px_origin, defocus_u, defocus_v;
    bool defocus = false;
    static Camera init(double vfov, double focus_dist, double defocus_angle, V3 look_from, V3 look_at, V3 vup,
                       size_t img_height, size_t img_width) {
        const double DEG_TO_RAD = 3.14159265358979323846264338327950288 / 180.0;
        const double fimg_h = (double)img_height, fimg_w = (double)img_width;
        const double vp_height = 2 * std::tan(vfov * DEG_TO_RAD / 2.0) * focus_dist;
        const double vp_width = vp_height * fimg_w / fimg_h;
        const V3 w = look_from.sub(look_at).unit();
        const V3 u = vup.cross(w).unit();
        const V3 v = w.cross(u);
        const V3 vp_u = u.mul(vp_width), vp_v = v.mul(-vp_height);
        const V3 px_du = vp_u.div(fimg_w), px_dv = vp_v.div(fimg_h);
        const double defocus_radius = std::tan(defocus_angle * DEG_TO_RAD / 2) * focus_dist;
        Camera c;
        c.look_from = look_from;
        c.px_du = px_du;
        c.px_dv = px_dv;
        c.px_origin = look_from.sub(w.mul(focus_dist)).sub(vp_u.div(2)).sub(vp_v.div(2)).add(px_du.add(px_dv).mul(0.5));
        c.defocus_u = u.mul(defocus_radius);
        c.defocus_v = v.mul(defocus_radius);
        c.defocus = defocus_angle > 0;
        return c;
    }
    RzCamera flat() const {
        RzCamera r;
        std::memset(&r, 0, sizeof r);
        auto put = [](double *d, V3 v) { d[0] = v.x; d[1] = v.y; d[2] = v.z; };
        put(r.look_from, look_from); put(r.px_du, px_du); put(r.px_dv, px_dv); put(r.px_origin, px_origin);
        put(r.defocus_u, defocus_u); put(r.defocus_v, defocus_v);
        r.defocus = defocus ? 1 : 0;
        return r;
    }
};

template <class T> struct Handle { size_t idx; };

struct Texture {
    enum Kind { checker = RZ_TEX_CHECKER, solid = RZ_TEX_SOLID } kind = solid;
    V3 color;                       // SolidTexture
    double scale = 1;               // CheckerTexture
    Handle<Texture> even{0}, odd{0};
    static Texture Solid(V3 c) { Texture t; t.kind = solid; t.color = c; return t; }
    static Texture Checker(double scale, Handle<Texture> even, Handle<Texture> odd) {
        Texture t; t.kind = checker; t.scale = scale; t.even = even; t.odd = odd; return t;
    }
};
using TextureHandle = Handle<Texture>;

struct Material {
    enum Kind { diffuse = RZ_MAT_DIFFUSE, metallic = RZ_MAT_METALLIC, dielectric = RZ_MAT_DIELECTRIC } kind = diffuse;
    uint32_t method = RZ_DIFFUSE_HEMISPHERE;  // material.zig:74
    double fuzz = 0, refractive_index = 1.0;
    TextureHandle texture{0};
    static Material Diffuse(TextureHandle t) { Material m; m.kind = diffuse; m.texture = t; return m; }
    static Material Metallic(TextureHandle t, double fuzz = 0) { Material m; m.kind = metallic; m.texture = t; m.fuzz = fuzz; return m; }
    static Material Dielectric(double ri) { Material m; m.kind = dielectric; m.refractive_index = ri; return m; }
};
using MaterialHandle = Handle<Material>;

struct Sphere {
    Ray center;
    double radius = 0;
    MaterialHandle material{0};
    static Sphere stationary(V3 c, double r, MaterialHandle m) { Sphere s; s.center.origin = c; s.center.dir = {}; s.radius = r; s.material = m; return s; }
};

struct MemPool {
    std::vector<Sphere> spheres;
    std::vector<Material> materials;
    std::vector<Texture> textures;
    void add(const Sphere &s) { spheres.push_back(s); }
    TextureHandle addAndReturnHandle(const Texture &t) { textures.push_back(t); return {textures.size() - 1}; }
    MaterialHandle addAndReturnHandle(const Material &m) { materials.push_back(m); return {materials.size() - 1}; }
    Handle<Sphere> addAndReturnHandle(const Sphere &s) { spheres.push_back(s); return {spheres.size() - 1}; }
};

struct Image {
    size_t h = 0, w = 0;
    std::vector<V3> pixels;        // linear radiance, pixels[j*w+i]  (image.zig:7)
    std::vector<uint8_t> rgb8;     // device-side sqrt/clamp/trunc of image.zig:35-38
    static Image initEmpty(size_t h, size_t w) { Image i; i.h = h; i.w = w; i.pixels.resize(h * w); return i; }
    // writePPM (image.zig:29-41): ASCII P3, "{r} {g} {b}\n" per pixel — the same bytes as the reference's writer.  At GPU
    // speed this text dump is the slowest step after the render (config 3: 8.3 M pixels, ~95 MB of text), so it is built for
    // throughput: one pre-sized buffer (at most 12 bytes per pixel), a table of the 256 possible "ddd " tokens copied as one
    // 32-bit word each, and a single fwrite.  Returns the number of bytes written.
    size_t formatPPM(std::vector<char> &buf) const {
        struct Tok { uint32_t word; uint32_t len; };   // up to 3 digits + separator, little-endian in one word
        static Tok sp[256], nl[256];
        static bool init = false;
        if (!init) {
            for (int v = 0; v < 256; v++) {
                char t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                const int n = std::snprintf(t, sizeof t, "%d", v);
                t[n] = ' ';
                std::memcpy(&sp[v].word, t, 4); sp[v].len = (uint32_t)n + 1u;
                t[n] = '\n';
                std::memcpy(&nl[v].word, t, 4); nl[v].len = (uint32_t)n + 1u;
            }
            init = true;
        }
        char head[64];
        const int hn = std::snprintf(head, sizeof head, "P3\n%zu %zu\n%d\n", w, h, 255);
        buf.resize((size_t)hn + h * w * 12 + 8);
        char *o = buf.data();
        std::memcpy(o, head, (size_t)hn);
        o += hn;
        const uint8_t *px = rgb8.data();
        for (size_t p = 0, n = h * w; p < n; p++, px += 3) {
            const Tok a = sp[px[0]], b = sp[px[1]], c = nl[px[2]];
            std::memcpy(o, &a.word, 4); o += a.len;     // 4-byte stores that overlap by up to 2 bytes: no per-byte loop
            std::memcpy(o, &b.word, 4); o += b.len;
            std::memcpy(o, &c.word, 4); o += c.len;
        }
        return (size_t)(o - buf.data());
    }
    size_t writePPM(FILE *f) const {
        std::vector<char> buf;
        const size_t n = formatPPM(buf);
        return std::fwrite(buf.data(), 1, n, f);
    }
};

struct CudaBackendError : std::runtime_error {
    int code;
    CudaBackendError(int c, const char *msg) : std::runtime_error(msg), code(c) {}
};

constexpr double ASPECT_RATIO = 16.0 / 9.0;  // renderer.zig:16

struct Tracer {
    Camera camera;
    Image img;
    DefaultPrng rng;
    size_t max_bounces = 50;      // renderer.zig:23
    size_t samples_per_px = 10;   // renderer.zig:24
    MemPool pool;
    // backend knobs (not in the reference)
    uint64_t render_seed = 1;
    uint32_t variant = RZ_VARIANT_AUTO;
    std::vector<int> devices{0};
    RzContext *ctx = nullptr;
    RzTiming timing{};
    float noise_target = 0;       // > 0: render from samples_per_px, doubling, until the frame's rms error reaches it (rayz_cuda_render_to_noise)
    uint32_t max_spp = 4096;      // ... or this many samples are in
    RzNoise noise{};              // summary of the last render with a noise target

    Tracer(size_t img_w, double vfov, double focus_dist, double defocus_angle, V3 look_from, V3 look_at, V3 vup, uint64_t seed)
        : rng(seed) {
        const size_t height = (size_t)((double)img_w / ASPECT_RATIO);  // renderer.zig:39-40
        camera = Camera::init(vfov, focus_dist, defocus_angle, look_from, look_at, vup, height, img_w);
        img = Image::initEmpty(height, img_w);
    }
    ~Tracer() { if (ctx) rayz_cuda_destroy(ctx); }
    Tracer(const Tracer &) = delete;
    Tracer &operator=(const Tracer &) = delete;

    static void check(int rc) { if (rc != RZ_OK) throw CudaBackendError(rc, rayz_cuda_last_error()); }

    // renderer.zig:72-101.  Returns the number of primary rays traced (`!usize`).
    // Device selection, CUDA context and kernel loading: the counterpart of the allocations
    // Tracer.init does before main starts its timer (renderer.zig:29-64, rayz.zig:22-24).
    void initBackend() {
        if (ctx) return;
        RzConfig cfg;
        std::memset(&cfg, 0, sizeof cfg);
        cfg.n_devices = (int32_t)devices.size();
        for (size_t i = 0; i < devices.size() && i < 8; i++) cfg.device_ids[i] = devices[i];
        check(rayz_cuda_create(&cfg, &ctx));
        const RzRenderParams p = renderParams();
        check(rayz_cuda_reserve(ctx, &p));   // like Image.initEmpty in Tracer.init: before the timer
    }

    RzRenderParams renderParams() const {
        RzRenderParams p;
        std::memset(&p, 0, sizeof p);
        p.width = (uint32_t)img.w; p.height = (uint32_t)img.h; p.spp = (uint32_t)samples_per_px; p.max_depth = (uint32_t)max_bounces;
        p.seed = render_seed; p.variant = variant;
        return p;
    }

    // The flattened MemPool (RzScene field order), kept alive here so that main can dump it (--dump-scene)
    std::vector<double> sc, sv, sr, mf, mi, tcol, ts;
    std::vector<uint32_t> sm, mk, mt, mm, tk, te, to;
    std::vector<float> lin;   // linear float4 frame of the last render (--dump-linear)

    size_t render() {
        initBackend();
        // pool.initHittables + bvh.build (:76-78) -> flatten + upload
        const size_t ns = pool.spheres.size(), nm = pool.materials.size(), nt = pool.textures.size();
        sc.assign(3 * ns, 0); sv.assign(3 * ns, 0); sr.assign(ns, 0); mf.assign(nm, 0); mi.assign(nm, 0); tcol.assign(3 * nt, 0); ts.assign(nt, 0);
        sm.assign(ns, 0); mk.assign(nm, 0); mt.assign(nm, 0); mm.assign(nm, 0); tk.assign(nt, 0); te.assign(nt, 0); to.assign(nt, 0);
        for (size_t i = 0; i < ns; i++) {
            const Sphere &s = pool.spheres[i];
            sc[3 * i] = s.center.origin.x; sc[3 * i + 1] = s.center.origin.y; sc[3 * i + 2] = s.center.origin.z;
            sv[3 * i] = s.center.dir.x; sv[3 * i + 1] = s.center.dir.y; sv[3 * i + 2] = s.center.dir.z;
            sr[i] = s.radius; sm[i] = (uint32_t)s.material.idx;
        }
        for (size_t i = 0; i < nm; i++) {
            const Material &m = pool.materials[i];
            mk[i] = m.kind; mf[i] = m.fuzz; mi[i] = m.refractive_index; mt[i] = (uint32_t)m.texture.idx; mm[i] = m.method;
        }
        for (size_t i = 0; i < nt; i++) {
            const Texture &t = pool.textures[i];
            tk[i] = t.kind; tcol[3 * i] = t.color.x; tcol[3 * i + 1] = t.color.y; tcol[3 * i + 2] = t.color.z;
            ts[i] = t.scale; te[i] = (uint32_t)t.even.idx; to[i] = (uint32_t)t.odd.idx;
        }
        RzScene s;
        std::memset(&s, 0, sizeof s);
        s.n_spheres = (uint32_t)ns; s.n_materials = (uint32_t)nm; s.n_textures = (uint32_t)nt;
        s.sphere_center = sc.data(); s.sphere_velocity = sv.data(); s.sphere_radius = sr.data(); s.sphere_material = sm.data();
        s.mat_kind = mk.data(); s.mat_fuzz = mf.data(); s.mat_ior = mi.data(); s.mat_texture = mt.data(); s.mat_method = mm.data();
        s.tex_kind = tk.data(); s.tex_color = tcol.data(); s.tex_scale = ts.data(); s.tex_even = te.data(); s.tex_odd = to.data();
        check(rayz_cuda_upload_scene(ctx, &s));

        const RzRenderParams p = renderParams();
        const RzCamera cam = camera.flat();
        lin.assign(img.w * img.h * 4, 0.f);
        img.rgb8.resize(img.w * img.h * 3);
        uint64_t rays = 0;
        if (noise_target > 0) check(rayz_cuda_render_to_noise(ctx, &cam, &p, noise_target, max_spp, lin.data(), img.rgb8.data(), &rays, &noise));
        else check(rayz_cuda_render(ctx, &cam, &p, lin.data(), img.rgb8.data(), &rays));
        for (size_t i = 0; i < img.w * img.h; i++) img.pixels[i] = {lin[4 * i], lin[4 * i + 1], lin[4 * i + 2]};
        rayz_cuda_timing(ctx, &timing);
        return (size_t)rays;
    }
};

// --dump-scene: the flattened scene as raw little-endian arrays in RzScene field order, each preceded by nothing — sizes
// follow from the three counts in the 16-byte header (n_spheres, n_materials, n_textures, 0).  Read by tests/test_host_gpu.py.
inline bool dumpScene(const Tracer &t, const char *path) {
    FILE *f = std::fopen(path, "wb");
    if (!f) return false;
    const uint32_t head[4] = {(uint32_t)t.sr.size(), (uint32_t)t.mk.size(), (uint32_t)t.tk.size(), 0u};
    std::fwrite(head, sizeof head, 1, f);
    auto d = [&](const std::vector<double> &v) { if (!v.empty()) std::fwrite(v.data(), sizeof(double), v.size(), f); };
    auto u = [&](const std::vector<uint32_t> &v) { if (!v.empty()) std::fwrite(v.data(), sizeof(uint32_t), v.size(), f); };
    d(t.sc); d(t.sv); d(t.sr); u(t.sm); u(t.mk); d(t.mf); d(t.mi); u(t.mt); u(t.mm); u(t.tk); d(t.tcol); d(t.ts); u(t.te); u(t.to);
    std::fclose(f);
    return true;
}

// rayz.zig:170-239 (dead code in the reference: it targets a removed MemPool API), in its insertion order
inline void penultimateScene(Tracer &tracer) {
    MemPool &pool = tracer.pool;
    pool.add(Sphere::stationary({0, 0, -1.2}, 0.5, pool.addAndReturnHandle(Material::Diffuse(pool.addAndReturnHandle(Texture::Solid({0.1, 0.2, 0.5}))))));
    pool.add(Sphere::stationary({0, -100.5, -1}, 100, pool.addAndReturnHandle(Material::Diffuse(pool.addAndReturnHandle(Texture::Solid({0.8, 0.8, 0.0}))))));
    pool.add(Sphere::stationary({-1, 0, -1}, 0.5, pool.addAndReturnHandle(Material::Dielectric(1.5))));         // left outer
    pool.add(Sphere::stationary({-1, 0, -1}, 0.4, pool.addAndReturnHandle(Material::Dielectric(1.0 / 1.5))));   // left inner bubble
    pool.add(Sphere::stationary({1, 0, -1}, 0.5, pool.addAndReturnHandle(Material::Metallic(pool.addAndReturnHandle(Texture::Solid({0.8, 0.6, 0.2})), 1.0))));
}

// rayz.zig:45-168
inline void randomBouncing(Tracer &tracer, int grid_lo = -11, int grid_hi = 11) {
    MemPool &pool = tracer.pool;
    DefaultPrng &rand = tracer.rng;
    // rayz.zig:57-73: Zig evaluates the nested struct literals in source order — even, odd, then the checker.  (C++ leaves the
    // order of function arguments unspecified, so the handles are taken one statement at a time: tests/test_host_gpu.py compares
    // the flattened scene with the oracle's byte for byte.)
    const TextureHandle even = pool.addAndReturnHandle(Texture::Solid({0.2, 0.3, 0.1}));
    const TextureHandle odd = pool.addAndReturnHandle(Texture::Solid(V3::of(0.9)));
    const TextureHandle checker = pool.addAndReturnHandle(Texture::Checker(0.32, even, odd));
    pool.add(Sphere::stationary({0, -1000, 0}, 1000, pool.addAndReturnHandle(Material::Diffuse(checker))));
    pool.add(Sphere::stationary({0, 1, 0}, 1.0, pool.addAndReturnHandle(Material::Dielectric(1.5))));
    pool.add(Sphere::stationary({-4, 1, 0}, 1.0, pool.addAndReturnHandle(Material::Diffuse(pool.addAndReturnHandle(Texture::Solid({0.4, 0.2, 0.1}))))));
    pool.add(Sphere::stationary({4, 1, 0}, 1.0, pool.addAndReturnHandle(Material::Metallic(pool.addAndReturnHandle(Texture::Solid({0.7, 0.6, 0.5}))))));
    for (int a = grid_lo; a < grid_hi; a++) {
        for (int b = grid_lo; b < grid_hi; b++) {
            const double rand_mat = rand.float64();
            V3 center;
            center.x = (double)a + 0.9 * rand.float64();
            center.y = 0.2;
            center.z = (double)b + 0.9 * rand.float64();
            if (center.sub({4, 0.2, 0}).mag() <= 0.9) continue;
            Ray sphere_ray;
            sphere_ray.origin = center;
            MaterialHandle m{0};
            if (rand_mat < 0.8) {
                const V3 c1 = rand.v3(0, 1.0);
                const V3 c2 = rand.v3(0, 1.0);
                m = pool.addAndReturnHandle(Material::Diffuse(pool.addAndReturnHandle(Texture::Solid(c1.vmul(c2)))));
                sphere_ray.dir = V3::y_hat().mul(rand.float64() * 0.5);
            } else if (rand_mat < 0.95) {
                const double fuzz = rand.float64() * 0.5;
                const V3 col = rand.v3(0.5, 1.0);
                m = pool.addAndReturnHandle(Material::Metallic(pool.addAndReturnHandle(Texture::Solid(col)), fuzz));
            } else {
                m = pool.addAndReturnHandle(Material::Dielectric(1.5));
            }
            Sphere s;
            s.center = sphere_ray;
            s.radius = 0.2;
            s.material = m;
            pool.add(s);
        }
    }
}

}  // namespace rayz
