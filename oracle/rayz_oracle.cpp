// rayz_oracle.cpp — CPU (f64) restatement of the rayz hot path.
//
// *** TEST INFRASTRUCTURE ONLY. ***  Nothing under rayz_b200/, host/ or include/ may include,
// link, load or execute this file.  Only tests/, __graft_entry__.smoke() and bench.py's
// cpu_baseline / --impl reference legs use it, and only as the checker / CPU baseline.
//
// The reference (jlucier/rayz, Zig) cannot be compiled here (no zig toolchain), so this file
// restates its algorithm function by function; every function cites the reference lines it
// follows (paths relative to /root/reference/src).  Build with -ffp-contract=off: Zig's default
// float mode is strict (no FMA fusion).
//
// Pinning: checked against every KAT the reference's own tests hold for this path
// (vec.zig:169-215, utils.zig:15-32, geom.zig:69-84, hit.zig:237-279, material.zig:213-223,
// renderer.zig:129-149) by tests/test_oracle_kat.py.  NOT pinned by any reference test (the
// reference has none): sphere hit, BVH, scatter, sky, render, quantise, scene generation, and
// the PRNG stream (Zig std is un-vendored and unversioned; Xoshiro256++/SplitMix64/float(f64)
// below restate Zig std 0.13's std.Random from its published algorithm).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <thread>
#include <vector>

namespace {

const double INF = std::numeric_limits<double>::infinity();

// ---------------------------------------------------------------- utils.zig:3-13
inline double u_min(double a, double b) { return a < b ? a : b; }
inline double u_max(double a, double b) { return a > b ? a : b; }
inline double u_clamp(double x, double lo, double hi) { return u_min(u_max(x, lo), hi); }

// ---------------------------------------------------------------- vec.zig:4-157
struct V3 {
    double x = 0, y = 0, z = 0;
    double at(int axis) const { return axis == 0 ? x : (axis == 1 ? y : z); }   // vec.zig:26-33
    V3 add(V3 o) const { return {x + o.x, y + o.y, z + o.z}; }                  // :47-53
    V3 sub(V3 o) const { return {x - o.x, y - o.y, z - o.z}; }                  // :55-61
    V3 mul(double v) const { return {x * v, y * v, z * v}; }                    // :63-65
    V3 div(double v) const { return mul(1 / v); }                               // :67-69 (reciprocal!)
    double dot(V3 o) const { return x * o.x + y * o.y + z * o.z; }              // :95-97
    double mag() const { return std::sqrt(dot(*this)); }                        // :71-73
    V3 unit() const { return div(mag()); }                                      // :75-77
    V3 clamp(double lo, double hi) const {                                      // :79-85
        return {u_clamp(x, lo, hi), u_clamp(y, lo, hi), u_clamp(z, lo, hi)};
    }
    V3 sqrt() const {                                                           // :87-93
        return {x > 0 ? std::sqrt(x) : 0, y > 0 ? std::sqrt(y) : 0, z > 0 ? std::sqrt(z) : 0};
    }
    V3 cross(V3 o) const {                                                      // :99-105
        return {y * o.z - z * o.y, z * o.x - x * o.z, x * o.y - y * o.x};
    }
    bool nearZero() const {                                                     // :107-110
        const double tol = 1e-8;
        return std::fabs(x) <= tol && std::fabs(y) <= tol && std::fabs(z) <= tol;
    }
    bool close(V3 o) const { return sub(o).nearZero(); }                        // :112-114
    V3 vmul(V3 o) const { return {x * o.x, y * o.y, z * o.z}; }                 // :118-124
    V3 vdiv(V3 o) const { return {x / o.x, y / o.y, z / o.z}; }                 // :126-132
    // @min/@max on floats return the non-NaN operand, like fmin/fmax          // :134-148
    V3 vmin(V3 o) const { return {std::fmin(x, o.x), std::fmin(y, o.y), std::fmin(z, o.z)}; }
    V3 vmax(V3 o) const { return {std::fmax(x, o.x), std::fmax(y, o.y), std::fmax(z, o.z)}; }
    int amax() const {                                                          // :150-156
        if (x > y) return x > z ? 0 : 2;
        return y > z ? 1 : 2;
    }
    static V3 of(double v) { return {v, v, v}; }
};

struct Ray {                                                                    // vec.zig:159-167
    V3 origin, dir;
    double time = 0;
    V3 at(double t) const { return origin.add(dir.mul(t)); }
};

// ---------------------------------------------------------------- Zig std.Random (un-vendored)
// DefaultPrng = Xoshiro256 (xoshiro256++), state = 4 SplitMix64 outputs of the seed;
// Random.float(f64): 52 mantissa bits, exponent 1022 - clz(top 12 bits) with refill.
struct Rng {
    uint64_t s[4];
    explicit Rng(uint64_t seed) {
        uint64_t sm = seed;
        for (int i = 0; i < 4; i++) {
            sm += 0x9e3779b97f4a7c15ull;
            uint64_t z = sm;
            z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
            z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
            s[i] = z ^ (z >> 31);
        }
    }
    static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
    uint64_t next() {
        const uint64_t r = rotl(s[0] + s[3], 23) + s[0];
        const uint64_t t = s[1] << 17;
        s[2] ^= s[0];
        s[3] ^= s[1];
        s[1] ^= s[2];
        s[0] ^= s[3];
        s[2] ^= t;
        s[3] = rotl(s[3], 45);
        return r;
    }
    static int clz64(uint64_t v) { return v == 0 ? 64 : __builtin_clzll(v); }
    double f64() {
        const uint64_t rand = next();
        uint64_t rand_lz = (uint64_t)clz64(rand);
        if (rand_lz >= 12) {
            rand_lz = 12;
            while (true) {
                const uint64_t addl = (uint64_t)clz64(next());
                rand_lz += addl;
                if (addl != 64) break;
                if (rand_lz >= 1022) { rand_lz = 1022; break; }
            }
        }
        const uint64_t mantissa = rand & 0xFFFFFFFFFFFFFull;
        const uint64_t exponent = (1022 - rand_lz) << 52;
        const uint64_t bits = exponent | mantissa;
        double d;
        std::memcpy(&d, &bits, 8);
        return d;
    }
    V3 v3(double low, double high) {                                            // vec.zig:9-16
        const double scale = high - low;
        V3 r;
        r.x = f64() * scale + low;
        r.y = f64() * scale + low;
        r.z = f64() * scale + low;
        return r;
    }
};

// ---------------------------------------------------------------- camera.zig:9-90
struct Camera {
    V3 look_from, px_du, px_dv, px_origin, defocus_u, defocus_v;
    bool defocus = false;

    static Camera init(double vfov, double focus_dist, double defocus_angle, V3 look_from,
                       V3 look_at, V3 vup, size_t img_height, size_t img_width) {  // :18-57
        const double DEG_TO_RAD = 3.14159265358979323846264338327950288 / 180.0;  // :7
        const double fimg_h = (double)img_height;
        const double fimg_w = (double)img_width;
        const double vp_height = 2 * std::tan(vfov * DEG_TO_RAD / 2.0) * focus_dist;
        const double vp_width = vp_height * fimg_w / fimg_h;
        const V3 w = look_from.sub(look_at).unit();
        const V3 u = vup.cross(w).unit();
        const V3 v = w.cross(u);
        const V3 vp_u = u.mul(vp_width);
        const V3 vp_v = v.mul(-vp_height);
        const V3 px_du = vp_u.div(fimg_w);
        const V3 px_dv = vp_v.div(fimg_h);
        const double defocus_radius = std::tan(defocus_angle * DEG_TO_RAD / 2) * focus_dist;
        const V3 vp_origin = look_from.sub(w.mul(focus_dist)).sub(vp_u.div(2)).sub(vp_v.div(2))
                                 .add(px_du.add(px_dv).mul(0.5));
        Camera c;
        c.look_from = look_from;
        c.px_du = px_du;
        c.px_dv = px_dv;
        c.px_origin = vp_origin;
        c.defocus_u = u.mul(defocus_radius);
        c.defocus_v = v.mul(defocus_radius);
        c.defocus = defocus_angle > 0;
        return c;
    }

    V3 randomInDefocus(Rng &rng) const {                                        // :79-90
        if (!defocus) return {};
        while (true) {
            V3 v;
            v.x = rng.f64() * 2 - 1;
            v.y = rng.f64() * 2 - 1;
            v.z = 0;
            if (v.dot(v) <= 1) return defocus_u.mul(v.x).add(defocus_v.mul(v.y));
        }
    }

    Ray getRay(size_t px, size_t py, Rng *rng) const {                          // :59-77
        double x = (double)px;
        double y = (double)py;
        V3 origin = look_from;
        if (rng) {
            x += rng->f64() - 0.5;
            y += rng->f64() - 0.5;
            origin = origin.add(randomInDefocus(*rng));
        }
        Ray r;
        // struct-literal fields evaluate in source order: dir, origin, time
        r.dir = px_du.mul(x).add(px_dv.mul(y)).add(px_origin).sub(origin);
        r.origin = origin;
        r.time = rng ? rng->f64() : 0;
        return r;
    }
};

// ---------------------------------------------------------------- hit.zig:16-99
struct Hit {
    V3 point, normal;
    double t = 0, u = 0, v = 0;
    bool front_face = false;
    uint32_t material = 0;
    int32_t sphere = -1;  // not in the reference (hit.zig:16-24); carried for the id parity check
    static Hit init(const Ray &ray, V3 point, V3 normal, double t, uint32_t material) {  // :25-41
        Hit h;
        h.front_face = normal.dot(ray.dir) < 0;
        h.point = point;
        h.normal = h.front_face ? normal : normal.mul(-1);
        h.t = t;
        h.material = material;
        return h;
    }
};

struct AABB {
    V3 low = V3::of(INF), high = V3::of(-INF);                                  // :45-46
    static AABB init(V3 a, V3 b) { AABB r; r.low = a.vmin(b); r.high = a.vmax(b); return r; }  // :48-53
    static AABB enclose(const AABB &a, const AABB &b) {                         // :55-60
        AABB r; r.low = a.low.vmin(b.low); r.high = a.high.vmax(b.high); return r;
    }
    int longestAxis() const { return high.sub(low).amax(); }                    // :62-64
    bool hit(const Ray &ray, double tmin, double tmax) const {                  // :70-98
        const V3 t0s = low.sub(ray.origin).vdiv(ray.dir);
        const V3 t1s = high.sub(ray.origin).vdiv(ray.dir);
        double t0 = tmin, t1 = tmax;
        for (int ax = 0; ax < 3; ax++) {
            const double v0 = t0s.at(ax), v1 = t1s.at(ax);
            if (v0 < v1) {
                t0 = std::fmax(v0, t0);
                t1 = std::fmin(v1, t1);
            } else {
                t0 = std::fmax(v1, t0);
                t1 = std::fmin(v0, t1);
            }
        }
        return t1 > t0;
    }
};

// ---------------------------------------------------------------- geom.zig:11-66
struct Sphere {
    Ray center;
    double radius = 0;
    uint32_t material = 0;
    AABB boundingBox() const {                                                  // :24-31
        const V3 rad = V3::of(radius);
        const V3 o1 = center.origin;
        const V3 o2 = center.at(1);
        return AABB::enclose(AABB::init(o1.sub(rad), o1.add(rad)), AABB::init(o2.sub(rad), o2.add(rad)));
    }
    bool hit(const Ray &ray, double tmin, double tmax, Hit &out) const {        // :38-66
        const V3 origin_now = center.at(ray.time);
        const V3 offset = origin_now.sub(ray.origin);
        const double a = ray.dir.dot(ray.dir);
        const double half_b = ray.dir.dot(offset);
        const double c = offset.dot(offset) - radius * radius;
        const double discriminant = half_b * half_b - a * c;
        if (discriminant < 0) return false;
        const double rt = std::sqrt(discriminant);
        const double t1 = (half_b - rt) / a;
        const double t2 = (half_b + rt) / a;
        double t;
        if (t1 >= tmin && t1 <= tmax) t = t1;
        else if (t2 >= tmin && t2 <= tmax) t = t2;
        else return false;
        const V3 point = ray.at(t);
        const V3 n = point.sub(origin_now).unit();
        out = Hit::init(ray, point, n, t, material);
        return true;
    }
};

// ---------------------------------------------------------------- material.zig:12-51, 162-211
struct Texture {
    uint32_t kind = 1;  // 0 checker, 1 solid (material.zig:41-43)
    V3 color;
    double scale = 1;
    uint32_t even = 0, odd = 0;
};
struct Material {
    uint32_t kind = 0;  // 0 diffuse, 1 metallic, 2 dielectric (material.zig:162-165)
    double fuzz = 0, ior = 1;
    uint32_t texture = 0;
    uint32_t method = 2;  // HEMISPHERE (material.zig:74)
};

struct Counters {
    uint64_t paths = 0, segments = 0, sphere_tests = 0, node_tests = 0;
    uint64_t hits[3] = {0, 0, 0};
    uint64_t ended_sky = 0, ended_absorbed = 0, ended_depth = 0;
    void add(const Counters &o) {
        paths += o.paths; segments += o.segments; sphere_tests += o.sphere_tests; node_tests += o.node_tests;
        for (int i = 0; i < 3; i++) hits[i] += o.hits[i];
        ended_sky += o.ended_sky; ended_absorbed += o.ended_absorbed; ended_depth += o.ended_depth;
    }
};

struct Hittable {  // hit.zig:8-12 (ptr+fn replaced by a sphere index)
    AABB bbox;
    uint32_t sphere;
};

struct BVHNode {  // hit.zig:101-108; children by index instead of pointer, same shape
    AABB bbox;
    size_t starti = 0, endi = 0;
    int left = -1, right = -1;
};

struct Scene {
    std::vector<Sphere> spheres;
    std::vector<Material> materials;
    std::vector<Texture> textures;
    std::vector<Hittable> hittables;
    std::vector<BVHNode> nodes;

    V3 textureValue(uint32_t idx, V3 point) const {                             // material.zig:20-50
        const Texture *t = &textures[idx];
        while (t->kind == 0) {  // CheckerTexture.value :32-38 (handle recursion → loop)
            const int64_t x = (int64_t)std::floor(point.x / t->scale);
            const int64_t y = (int64_t)std::floor(point.y / t->scale);
            const int64_t z = (int64_t)std::floor(point.z / t->scale);
            const int64_t s = x + y + z;
            const int64_t m = ((s % 2) + 2) % 2;  // @mod: floor-mod
            t = &textures[m == 0 ? t->even : t->odd];
        }
        return t->color;
    }

    void initHittables() {                                                      // ecs.zig:43-51
        hittables.clear();
        for (size_t i = 0; i < spheres.size(); i++) hittables.push_back({spheres[i].boundingBox(), (uint32_t)i});
    }
    int buildNode(size_t si, size_t ei) {                                       // hit.zig:130-161
        const int me = (int)nodes.size();
        nodes.push_back(BVHNode());
        AABB bb;
        for (size_t i = si; i < ei; i++) bb = AABB::enclose(bb, hittables[i].bbox);
        nodes[me].bbox = bb;
        const size_t nobjs = ei - si;
        if (nobjs <= 2) {
            nodes[me].starti = si;
            nodes[me].endi = ei;
        } else {
            const int axis = bb.longestAxis();
            std::stable_sort(hittables.begin() + si, hittables.begin() + ei,      // std.mem.sort is stable
                             [axis](const Hittable &a, const Hittable &b) { return a.bbox.low.at(axis) < b.bbox.low.at(axis); });
            const size_t mid = nobjs / 2 + si;
            const int l = buildNode(si, mid);
            const int r = buildNode(mid, ei);
            nodes[me].left = l;
            nodes[me].right = r;
        }
        return me;
    }
    void build() {                                                              // renderer.zig:76-78
        initHittables();
        nodes.clear();
        if (!hittables.empty()) buildNode(0, hittables.size());
    }

    bool findHit(int ni, const Ray &ray, double tmin, double tmax, Hit &out, Counters *c) const {  // hit.zig:181-216
        const BVHNode &n = nodes[ni];
        if (c) c->node_tests++;
        if (!n.bbox.hit(ray, tmin, tmax)) return false;
        bool have = false;
        if (n.left >= 0) {
            have = findHit(n.left, ray, tmin, tmax, out, c);
            const double maxt = have ? out.t : tmax;
            Hit nh;
            if (findHit(n.right, ray, tmin, maxt, nh, c)) { out = nh; have = true; }
            return have;
        }
        for (size_t i = n.starti; i < n.endi; i++) {
            const double maxt = have ? out.t : tmax;
            Hit nh;
            if (c) c->sphere_tests++;
            if (spheres[hittables[i].sphere].hit(ray, tmin, maxt, nh)) {
                nh.sphere = (int32_t)hittables[i].sphere;
                out = nh;
                have = true;
            }
        }
        return have;
    }
    // Brute force in pool order with the same shrinking-tmax rule (cross-check of the BVH).
    bool findHitBrute(const Ray &ray, double tmin, double tmax, Hit &out) const {
        bool have = false;
        for (size_t i = 0; i < spheres.size(); i++) {
            const double maxt = have ? out.t : tmax;
            Hit nh;
            if (spheres[i].hit(ray, tmin, maxt, nh)) { nh.sphere = (int32_t)i; out = nh; have = true; }
        }
        return have;
    }
};

V3 randomInUnitSphere(Rng &rng) {                                               // material.zig:196-202
    while (true) {
        const V3 v = rng.v3(-1, 1);
        if (v.mag() <= 1) return v;
    }
}
V3 randomUnit(Rng &rng) { return randomInUnitSphere(rng).unit(); }               // :204-206
V3 randomInHemisphere(Rng &rng, V3 norm) {                                      // :208-211
    const V3 r = randomInUnitSphere(rng);
    return r.dot(norm) > 0 ? r : r.mul(-1);
}
double reflectance(double cosv, double ri) {                                    // :179-183
    double r0 = (1 - ri) / (1 + ri);
    r0 *= r0;
    return r0 + (1 - r0) * std::pow(1 - cosv, 5);
}
V3 reflect(const Ray &ray, const Hit &hit) {                                    // :185-187
    return ray.dir.sub(hit.normal.mul(2 * ray.dir.dot(hit.normal)));
}
V3 refract(V3 unit_dir, V3 norm, double eta) {                                  // :189-194
    const double cos_theta = unit_dir.mul(-1).dot(norm);
    const V3 perp_comp = norm.mul(cos_theta).add(unit_dir).mul(eta);
    const V3 parallel_comp = norm.mul(-std::sqrt(1 - perp_comp.dot(perp_comp)));
    return perp_comp.add(parallel_comp);
}

struct ScatterResult { Ray ray; V3 attenuation; };

bool scatter(const Scene &sc, const Material &m, Rng &rng, const Ray &ray, const Hit &hit, ScatterResult &res) {
    if (m.kind == 0) {                                                          // DiffuseMaterial.scatter :77-101
        V3 target;
        if (m.method == 0) target = hit.point.add(hit.normal).add(randomInUnitSphere(rng));
        else if (m.method == 1) target = hit.point.add(hit.normal).add(randomUnit(rng));
        else target = hit.point.add(randomInHemisphere(rng, hit.normal));
        if (target.nearZero()) target = hit.normal;
        res.ray.origin = hit.point;
        res.ray.dir = target.sub(hit.point);
        res.ray.time = ray.time;
        res.attenuation = sc.textureValue(m.texture, hit.point);
        return true;
    }
    if (m.kind == 1) {                                                          // MetallicMaterial.scatter :108-131
        V3 reflection_dir = reflect(ray, hit).unit();
        if (m.fuzz > 0) reflection_dir = reflection_dir.add(randomUnit(rng).mul(std::fmin(m.fuzz, 1.0)));
        if (reflection_dir.dot(hit.normal) <= 0) return false;
        res.ray.origin = hit.point;
        res.ray.dir = reflection_dir;
        res.ray.time = ray.time;
        res.attenuation = sc.textureValue(m.texture, hit.point);
        return true;
    }
    // DielectricMaterial.scatter :137-159
    const double eta = hit.front_face ? 1 / m.ior : m.ior;
    const V3 unit_dir = ray.dir.unit();
    const double cos_theta = unit_dir.mul(-1).dot(hit.normal);
    const double sin_theta = std::sqrt(1 - cos_theta * cos_theta);
    V3 dir;
    // Zig `or` short-circuits: no PRNG draw under total internal reflection
    if (eta * sin_theta > 1.0 || reflectance(cos_theta, eta) > rng.f64()) dir = reflect(ray, hit);
    else dir = refract(unit_dir, hit.normal, eta);
    res.ray.origin = hit.point;
    res.ray.dir = dir;
    res.ray.time = ray.time;
    res.attenuation = V3::of(1);
    return true;
}

// ---------------------------------------------------------------- renderer.zig:103-126
V3 bounceRay(const Scene &sc, Rng &rng, const Ray &ray, size_t depth, bool brute, Counters *c) {
    if (depth == 0) { if (c) c->ended_depth++; return {}; }
    Hit hit;
    if (c) c->segments++;
    const bool have = brute ? sc.findHitBrute(ray, 1e-10, INF, hit) : sc.findHit(0, ray, 1e-10, INF, hit, c);
    if (have) {
        V3 ret;
        const Material &m = sc.materials[hit.material];
        if (c) c->hits[m.kind]++;
        ScatterResult res;
        if (scatter(sc, m, rng, ray, hit, res)) ret = bounceRay(sc, rng, res.ray, depth - 1, brute, c).vmul(res.attenuation);
        else if (c) c->ended_absorbed++;
        return ret;
    }
    if (c) c->ended_sky++;
    const double t = 0.5 * (ray.dir.unit().y + 1.0);
    V3 blue; blue.x = 0.5; blue.y = 0.7; blue.z = 1.0;
    return V3::of(1).mul(1.0 - t).add(blue).mul(t);   // NOT a lerp: ((1-t) + c) * t   (:124-125)
}

uint64_t splitmix(uint64_t x) {
    x += 0x9e3779b97f4a7c15ull;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

// Rows [j0,j1) of renderer.zig:80-97 with one sequential PRNG.
void renderRows(const Scene &sc, const Camera &cam, size_t w, size_t j0, size_t j1, size_t spp, size_t depth,
                Rng &rng, bool brute, double *out, Counters *c) {
    for (size_t j = j0; j < j1; j++) {
        for (size_t i = 0; i < w; i++) {
            V3 acc;
            for (size_t r = 0; r < spp; r++) {
                const Ray ray = cam.getRay(i, j, &rng);
                if (c) c->paths++;
                acc = acc.add(bounceRay(sc, rng, ray, depth, brute, c));
            }
            const V3 px = acc.div((double)spp);
            out[(j * w + i) * 3 + 0] = px.x;
            out[(j * w + i) * 3 + 1] = px.y;
            out[(j * w + i) * 3 + 2] = px.z;
        }
    }
}

struct OrcScene { Scene sc; };

// =====================================================================================
// Path replay: the CUDA backend's documented path algorithm restated in f64, drawing the same uniforms, so that every
// GPU path (seed, pixel, sample) can be compared with its f64 counterpart one by one (tests/test_replay_*.py).  Restated from
// the product's CONTRACT, not from its code: nothing here includes or links a product header.  Each step cites the contract
// lines it follows (rayz_b200/csrc/rz_device.cuh, rz_search.cuh, rz_sampler.cuh, include/rayz_cuda.h).
//
// Where the algorithm deliberately differs from the reference above (the reference's sequential PRNG, its 1e-10 t_min and
// epsilon-free self intersection, its rejection samplers) the replay follows the backend, because it checks the backend path
// by path; tests/test_replay_cpu.py checks that the replay agrees with Scene.render in distribution.
//
// Robustness.  The GPU path runs in f32, so a path whose f64 decisions sit within f32 rounding of a boundary may take the
// other branch there.  The replay marks a path fragile from the first decision within the margins below, and also replays
// it with its camera and scatter directions perturbed by +-REPLAY_PERTURB: a changed event sequence marks it fragile too,
// and the largest radiance change sets its tolerance.
// =====================================================================================
namespace replay {

// ---- margins (the f32 error model each comes from)
const double U32 = 5.9604644775390625e-08;   // 2^-24: unit roundoff of f32
// Lengths (sphere-test operands, roots, hit points): every f32 operand carries its own rounding (|centre|, |origin|, r) and
// the sphere test chains ~a dozen roundings of numbers of size |oc| (rz_sphere_test: fma chains of oc, nb, l): 16 u per scale.
const double K_POS = 16.0 * U32;
// Directions: the GPU's unit directions carry ~1e-6 rad of error (__sincosf of the scatter angles, rsqrtf normalisation,
// the f32 normal); not measured, so the margin takes four times that.
const double DIR_ERR = 4e-6;
// Dot products of two such directions (diffuse flip s.n, metal r.n, the 1e-3 self-out margin): both operands' errors.
const double DOT_TOL = 2.0 * DIR_ERR;
// Schlick(cos, eta) against u.x and eta sin against 1: |dSchlick/dcos| = 5 (1 - r0) m^4 <= 5, and eta sin moves by
// eta cos / sin dcos: a direction error of DIR_ERR moves both by at most ~5 DIR_ERR away from grazing.
const double FRESNEL_TOL = 5.0 * DIR_ERR;
// Perturbed replays: directions turned by this angle (ten times the GPU's ~1e-6 rad direction error: 4e-6 missed a path of
// the all-materials scene whose f32 error grew through reflections between spheres in contact), in antithetic pairs
// (the default of orc_replay's `perturb`).
const double REPLAY_PERTURB = 1e-5;
const int REPLAY_PAIRS = 2;
// Tolerance of a robust path's radiance: SAFETY x the largest change among its perturbed replays, plus the f32 rounding of
// the throughput product (two roundings per bounce: the f32 colour and the product) and of the sky, plus an absolute floor
// (the 2^-32 fixed point of the accumulators and the f32 output).
const double TOL_SAFETY = 4.0;
const double TOL_REL_PER_SEG = 8.0 * U32;
const double TOL_ABS = 1e-8;

enum Reason { R_NONE = 0, R_TIE, R_GRAZE, R_TMIN, R_SELF_B, R_FLIP, R_METAL, R_TIR, R_FRESNEL, R_SELF_OUT, R_CHECKER,
              R_DEGENERATE, R_PERTURB };
enum End { E_SKY = 0, E_ABSORBED = 1, E_DEPTH = 2 };

// ---- uniforms (rz_device.cuh:281-316 Philox4x32-7; rz_sampler.cuh Owen-scrambled Sobol, restated after the numpy model of
// tests/test_sampler_cpu.py)
void philox(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int i = 0; i < 7; i++) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t h0 = (uint32_t)(p0 >> 32), l0 = (uint32_t)p0, h1 = (uint32_t)(p1 >> 32), l1 = (uint32_t)p1;
        const uint32_t n0 = h1 ^ c[1] ^ k0, n2 = h0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = l1; c[2] = n2; c[3] = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
uint32_t brev(uint32_t x) { uint32_t r = 0; for (int b = 0; b < 32; b++) r |= ((x >> b) & 1u) << (31 - b); return r; }
uint32_t hash32(uint32_t x) { x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16; return x; }
uint32_t owen(uint32_t x, uint32_t seed) {
    x = brev(x) + seed;
    for (uint32_t c : {0x6c50b47cu, 0xb82f1e52u, 0xc7afe638u, 0x8d22f6e6u}) x ^= x * c;
    return brev(x);
}
uint32_t sobol_d1(uint32_t i) {   // Joe-Kuo d = 2: V_j = m_j << (31 - j), m_0 = 1, m_j = m_{j-1} ^ (m_{j-1} << 1)
    uint32_t m = 1, r = 0;
    for (int j = 0; j < 32; j++) {
        if ((i >> j) & 1u) r ^= m << (31 - j);
        m ^= m << 1;
    }
    return r;
}
// the pair's two uniforms, top 24 bits of each coordinate (include/rayz_cuda.h RZ_RENDER_SOBOL / RZ_RENDER_RQMC)
void sobol_pair(uint32_t k0, uint32_t k1, uint32_t gpix, uint32_t pair, uint32_t sample, bool rqmc, double out[2]) {
    uint32_t base = hash32(hash32(hash32(hash32(k0 ^ 0x6a09e667u) ^ k1) ^ gpix) ^ pair);
    if (rqmc) { base = hash32(base ^ (0x9e3779b9u + (sample & 1u))); sample >>= 1; }
    const uint32_t i = owen(sample, hash32(base));
    out[0] = (double)(owen(brev(i), hash32(base ^ 1u)) >> 8) * U32;
    out[1] = (double)(owen(sobol_d1(i), hash32(base ^ 2u)) >> 8) * U32;
}
struct Keys { uint32_t k0, k1, gpix, sample; int sampler; };   // sampler: 0 Philox, 1 Sobol, 2 Sobol-RQMC
// camera: ux, uy (jitter), ut (time), ur, ua (lens radius, angle)   (rz_device.cuh:456-472)
void camera_uniforms(const Keys &K, double u[5]) {
    if (K.sampler) {
        double j[2], l[2], t[2];
        sobol_pair(K.k0, K.k1, K.gpix, 0, K.sample, K.sampler == 2, j);
        sobol_pair(K.k0, K.k1, K.gpix, 1, K.sample, K.sampler == 2, l);
        sobol_pair(K.k0, K.k1, K.gpix, 2, K.sample, K.sampler == 2, t);
        u[0] = j[0]; u[1] = j[1]; u[2] = t[0]; u[3] = l[0]; u[4] = l[1];
        return;
    }
    uint32_t c[4] = {K.gpix, K.sample, 0u, 0u};
    philox(c, K.k0, K.k1);
    u[0] = (double)(c[0] >> 8) * U32; u[1] = (double)(c[1] >> 8) * U32; u[2] = (double)(c[2] >> 8) * U32; u[3] = (double)(c[3] >> 8) * U32;
    u[4] = (double)(((c[0] & 0xffu) << 16) | ((c[1] & 0xffu) << 8) | (c[2] & 0xffu)) * U32;
}
// bounce s (1-based): Philox counter (gpix, sample, s, 0); Sobol pair 2 + s replaces u.x, u.y   (rz_search.cuh:397-401)
void bounce_uniforms(const Keys &K, uint32_t s, double u[4]) {
    uint32_t c[4] = {K.gpix, K.sample, s, 0u};
    philox(c, K.k0, K.k1);
    for (int i = 0; i < 4; i++) u[i] = (double)(c[i] >> 8) * U32;
    if (K.sampler) sobol_pair(K.k0, K.k1, K.gpix, 2u + s, K.sample, K.sampler == 2, u);
}

// ---- one path
struct Params {
    const Scene *sc;
    Camera cam;
    uint32_t depth;
    double t_min;
    double perturb;       // direction perturbation of this replay (0: the nominal path)
    uint32_t pert_id;     // which perturbation (hash input)
};
struct Path {
    double rgb[3] = {0, 0, 0};
    uint32_t segs = 0, hits[3] = {0, 0, 0};
    int end = E_DEPTH;
    int reason = R_NONE, fseg = -1;        // first fragile decision and its segment (0 = camera segment)
    std::vector<uint64_t> ev;              // one event word per segment, then the end kind
};

V3 perturbed(V3 d, const Keys &K, const Params &P, uint32_t seg) {
    if (P.perturb == 0) return d;
    // a direction perpendicular to d from a hash of (path, segment, perturbation); antithetic pairs share it with opposite signs
    uint32_t h = hash32(hash32(hash32(K.gpix * 0x9e3779b9u ^ K.sample) ^ seg) ^ (P.pert_id >> 1));
    V3 e;
    e.x = (double)(h & 0xffff) / 65535.0 - 0.5; h = hash32(h);
    e.y = (double)(h & 0xffff) / 65535.0 - 0.5; h = hash32(h);
    e.z = (double)(h & 0xffff) / 65535.0 - 0.5;
    e = e.sub(d.mul(e.dot(d)));
    const double m = e.mag();
    if (!(m > 1e-9)) return d;
    const double s = (P.pert_id & 1u) ? -P.perturb : P.perturb;
    return d.add(e.mul(s / m)).unit();
}

void fragile(Path &p, int reason, uint32_t seg) {
    if (p.reason == R_NONE) { p.reason = reason; p.fseg = (int)seg; }
}

// Texture walk in f64 on the f64 hit point (rz_device.cuh:481-503): floor(p * (1 / scale)), floor-mod 2 of the sum.  Returns
// the final texture; `near_edge` is set when a lattice coordinate lies within `dp` (hit-point error) of a cell boundary.
uint32_t texture_at(const Scene &sc, uint32_t tex, V3 p, double dp, bool &near_edge) {
    for (int level = 0; level < 8 && sc.textures[tex].kind == 0; level++) {
        const Texture &t = sc.textures[tex];
        const double inv = 1.0 / t.scale;
        int64_t s = 0;
        for (int ax = 0; ax < 3; ax++) {
            const double x = p.at(ax) * inv, f = std::floor(x);
            if (x - f < dp * inv || f + 1.0 - x < dp * inv) near_edge = true;
            s += (int64_t)f;
        }
        tex = (s & 1) == 0 ? t.even : t.odd;
    }
    return tex;
}

// rz_uniform_sphere: z = 1 - 2 u1, angle (u2 - 0.5) 2 pi
V3 uniform_sphere(double u1, double u2) {
    const double z = 1.0 - 2.0 * u1, r = std::sqrt(std::fmax(0.0, 1.0 - z * z));
    const double a = (u2 - 0.5) * 6.283185307179586476925286766559;
    V3 v; v.x = r * std::cos(a); v.y = r * std::sin(a); v.z = z;
    return v;
}

uint64_t fnv(uint64_t h, uint64_t w) { for (int i = 0; i < 8; i++) { h ^= (w >> (8 * i)) & 0xffu; h *= 0x100000001b3ull; } return h; }

void trace(const Keys &K, uint32_t px, uint32_t py, const Params &P, Path &out) {
    const Scene &sc = *P.sc;
    const Camera &cam = P.cam;
    const uint32_t n = (uint32_t)sc.spheres.size();
    double cu[5];
    camera_uniforms(K, cu);
    // Camera (rz_lens_ray, rz_device.cuh:435-454): x = px + (ux - 0.5), y = py + (uy - 0.5); thin lens polar, radius sqrt(ur),
    // angle (ua - 0.5) 2 pi; dir = px_du x + px_dv y + px_origin - o, normalised; time = ut
    V3 o = cam.look_from;
    double o_err = 0;   // f32 error of the origin beyond its own representation: the lens offset's arithmetic
    if (cam.defocus) {
        const double rad = std::sqrt(cu[3]), a = (cu[4] - 0.5) * 6.283185307179586476925286766559;
        const V3 off = cam.defocus_u.mul(rad * std::cos(a)).add(cam.defocus_v.mul(rad * std::sin(a)));
        o = o.add(off);
        o_err = DIR_ERR * off.mag();
    }
    const double x = (double)px + (cu[0] - 0.5), y = (double)py + (cu[1] - 0.5);
    const V3 dir = cam.px_du.mul(x).add(cam.px_dv.mul(y)).add(cam.px_origin).sub(o);
    V3 d = dir.unit();
    d = perturbed(d, K, P, 0);
    // the f32 camera: its six vectors rounded, and the sum rounded at the size of its largest term
    double d_err = DIR_ERR + K_POS * (cam.px_du.mag() * std::fabs(x) + cam.px_dv.mag() * std::fabs(y) + cam.px_origin.mag() + o.mag()) / dir.mag();
    const double time = cu[2];
    int self = -1;
    bool self_out = false;
    V3 thr = V3::of(1.0);
    uint32_t seg = 0;
    // rz_path.cu:149 / rz_search.cuh:405: a depth-0 path ends at once, black, counted as ended_depth (renderer.zig:104-105)
    if (P.depth == 0) { out.end = E_DEPTH; out.ev.push_back(0xd0); return; }
    while (true) {
        // ---- closest hit over every sphere, centre moved to c + v time (rz_sphere_test, rz_consider: rz_device.cuh:404-433)
        const double o_scale = o.mag();
        double bt = INF, bt_err = 0, t2 = INF, t2_err = 0;
        int bk = -1;
        bool bfar = false;
        for (uint32_t k = 0; k < n; k++) {
            const Sphere &s = sc.spheres[k];
            const V3 C = s.center.origin.add(s.center.dir.mul(time));
            const V3 oc = C.sub(o);
            const double b = oc.dot(d);
            const V3 l = oc.sub(d.mul(b));
            const double r = s.radius, ll = l.mag();
            const double occ = oc.mag();
            // f32 error of the line test and of b: operand roundings at the scale of the numbers involved (the origin, oc, r),
            // plus the direction error over the distance b to the closest approach, plus the origin's own
            const double dl = K_POS * (o_scale + std::fmax(occ, r)) + d_err * std::fabs(b) + o_err;
            if (std::fabs(ll - r) < dl) fragile(out, R_GRAZE, seg);
            const double nd = ll * ll - r * r;   // the line meets the sphere iff nd < 0
            if (!(nd < 0)) continue;
            const double sq = std::sqrt(-nd);
            const double dt = dl * (1.0 + std::fmin(ll / std::fmax(sq, 1e-300), 1e6));   // roots: sq = sqrt(r^2 - |l|^2) amplifies
            double t;
            bool far = false;
            if ((int)k == self) {
                // the sphere the ray starts on: only the far root, only while b > 0, never after RZ_SELF_OUT
                if (self_out) continue;
                if (std::fabs(b) < dl) fragile(out, R_SELF_B, seg);
                if (!(b > 0)) continue;
                t = b + sq; far = true;
            } else {
                t = b - sq;
                if (std::fabs(t - P.t_min) < dt) fragile(out, R_TMIN, seg);
                if (!(t > P.t_min)) { t = b + sq; far = true; }
            }
            if (std::fabs(t - P.t_min) < dt) fragile(out, R_TMIN, seg);
            if (!(t > P.t_min)) continue;
            if (t < bt) { t2 = bt; t2_err = bt_err; bt = t; bt_err = dt; bk = (int)k; bfar = far; }
            else if (t < t2) { t2 = t; t2_err = dt; }
        }
        if (bk >= 0 && t2 < INF && t2 - bt < bt_err + t2_err) fragile(out, R_TIE, seg);
        if (bk < 0) {
            // ---- sky (rz_sky, rz_device.cuh:474-479): ((1 - t) + (0.5, 0.7, 1.0)) t, t = 0.5 (d.y + 1); clamp [0, 2^20]
            out.segs++;
            const double t = 0.5 * (d.y + 1.0), a = 1.0 - t;
            const double L[3] = {thr.x * (a + 0.5) * t, thr.y * (a + 0.7) * t, thr.z * (a + 1.0) * t};
            for (int c = 0; c < 3; c++) out.rgb[c] = std::fmin(std::fmax(L[c], 0.0), 1048576.0);
            out.end = E_SKY;
            out.ev.push_back(0x5c);
            return;
        }
        out.segs++;
        // ---- the hit, in f64 (rz_refine_hit, rz_device.cuh:512-546): normal flipped against the ray
        const Sphere &s = sc.spheres[bk];
        const Material &m = sc.materials[s.material];
        const V3 C = s.center.origin.add(s.center.dir.mul(time));
        const V3 p = o.add(d.mul(bt));
        V3 nrm = p.sub(C).mul(1.0 / s.radius);
        const bool front = nrm.dot(d) < 0;
        if (!front) nrm = nrm.mul(-1);
        out.hits[m.kind < 3 ? m.kind : 0]++;
        seg++;
        double uu[4];
        bounce_uniforms(K, seg, uu);
        // hit-point error: the ray's origin and direction errors, along the surface (1 / cos of the incidence)
        const double cosi = std::fmax(std::fabs(nrm.dot(d)), 1e-3);
        const double dp = (K_POS * o_scale + d_err * bt + o_err) / cosi + K_POS * p.mag();
        V3 nd;
        int branch;
        uint32_t tex_hit = 0xffffffffu;
        bool edge = false;
        // ---- scatter (rz_scatter, rz_device.cuh:566-613)
        if (m.kind == 0) {
            const V3 sdir = uniform_sphere(uu[0], uu[1]);
            if (m.method == 2) {
                const double sn = sdir.dot(nrm);
                if (std::fabs(sn) < DOT_TOL) fragile(out, R_FLIP, seg - 1);
                nd = sn > 0 ? sdir : sdir.mul(-1);
            } else {
                const double rad = m.method == 0 ? std::cbrt(uu[2]) : 1.0;
                V3 t = nrm.add(sdir.mul(rad));
                const double tt = t.dot(t);
                if (tt < 1e-10) fragile(out, R_DEGENERATE, seg - 1);
                if (tt < 1e-12) t = nrm;
                nd = t.unit();
            }
            tex_hit = texture_at(sc, m.texture, p, dp, edge);
            thr = thr.vmul(sc.textures[tex_hit].color);
            branch = 0;
        } else if (m.kind == 1) {
            V3 r = d.sub(nrm.mul(2.0 * d.dot(nrm)));
            if (m.fuzz > 0) r = r.add(uniform_sphere(uu[0], uu[1]).mul(std::fmin(m.fuzz, 1.0)));
            const double rn = r.dot(nrm);
            if (std::fabs(rn) < DOT_TOL * (1.0 + std::fmin(m.fuzz, 1.0))) fragile(out, R_METAL, seg - 1);
            if (!(rn > 0)) {
                out.end = E_ABSORBED;
                out.ev.push_back(fnv(fnv(0xcbf29ce484222325ull, (uint64_t)bk * 2 + (bfar ? 1 : 0)), 0xab));
                out.ev.push_back(0xab);
                return;
            }
            nd = r.unit();
            tex_hit = texture_at(sc, m.texture, p, dp, edge);
            thr = thr.vmul(sc.textures[tex_hit].color);
            branch = 1;
        } else {
            const double ior = m.ior;
            const double eta = front ? 1.0 / ior : ior;
            const double cos_t = std::fmin(-d.dot(nrm), 1.0);
            const double sin_t = std::sqrt(std::fmax(0.0, 1.0 - cos_t * cos_t));
            double r0 = (1.0 - eta) / (1.0 + eta);
            r0 *= r0;
            const double mm = 1.0 - cos_t;
            const double schlick = r0 + (1.0 - r0) * (mm * mm * mm * mm * mm);
            if (std::fabs(eta * sin_t - 1.0) < FRESNEL_TOL) fragile(out, R_TIR, seg - 1);
            const bool tir = eta * sin_t > 1.0;
            if (!tir && std::fabs(schlick - uu[0]) < FRESNEL_TOL) fragile(out, R_FRESNEL, seg - 1);
            if (tir || schlick > uu[0]) {
                nd = d.sub(nrm.mul(2.0 * d.dot(nrm)));
                branch = tir ? 2 : 3;
            } else {
                const V3 perp = d.add(nrm.mul(cos_t)).mul(eta);
                const double par = -std::sqrt(std::fmax(0.0, 1.0 - perp.dot(perp)));
                nd = perp.add(nrm.mul(par));
                branch = 4;
            }
            nd = nd.unit();
        }
        if (edge) fragile(out, R_CHECKER, seg - 1);
        out.ev.push_back(fnv(fnv(fnv(0xcbf29ce484222325ull, (uint64_t)bk * 2 + (bfar ? 1 : 0)), (uint64_t)branch), tex_hit));
        nd = perturbed(nd, K, P, seg);
        // RZ_SELF_OUT: the ray leaves its sphere outward by more than 1e-3 (rz_device.cuh:609-611); time is kept
        const double outd = nd.dot(nrm), so = front ? outd : -outd;
        if (std::fabs(so - 1e-3) < DOT_TOL) fragile(out, R_SELF_OUT, seg - 1);
        self_out = so > 1e-3;
        self = bk;
        o = p;
        o_err = 0;
        d_err = DIR_ERR;
        d = nd;
        if (seg >= P.depth) { out.end = E_DEPTH; out.ev.push_back(0xd0); return; }   // rz_search.cuh:405
    }
}

}  // namespace replay

}  // namespace

// =====================================================================================
// C API (ctypes).  Flat scene layout == RzScene of include/rayz_cuda.h.
// =====================================================================================
extern "C" {

struct OrcCamera {  // == RzCamera
    double look_from[3], px_du[3], px_dv[3], px_origin[3], defocus_u[3], defocus_v[3];
    int32_t defocus, reserved0;
};

static Camera toCam(const OrcCamera *c) {
    Camera k;
    k.look_from = {c->look_from[0], c->look_from[1], c->look_from[2]};
    k.px_du = {c->px_du[0], c->px_du[1], c->px_du[2]};
    k.px_dv = {c->px_dv[0], c->px_dv[1], c->px_dv[2]};
    k.px_origin = {c->px_origin[0], c->px_origin[1], c->px_origin[2]};
    k.defocus_u = {c->defocus_u[0], c->defocus_u[1], c->defocus_u[2]};
    k.defocus_v = {c->defocus_v[0], c->defocus_v[1], c->defocus_v[2]};
    k.defocus = c->defocus != 0;
    return k;
}
static void put3(double *d, V3 v) { d[0] = v.x; d[1] = v.y; d[2] = v.z; }

void orc_camera_init(double vfov, double focus_dist, double defocus_angle, const double *from, const double *at,
                     const double *up, uint64_t img_h, uint64_t img_w, OrcCamera *out) {
    const Camera c = Camera::init(vfov, focus_dist, defocus_angle, {from[0], from[1], from[2]}, {at[0], at[1], at[2]},
                                  {up[0], up[1], up[2]}, (size_t)img_h, (size_t)img_w);
    put3(out->look_from, c.look_from); put3(out->px_du, c.px_du); put3(out->px_dv, c.px_dv);
    put3(out->px_origin, c.px_origin); put3(out->defocus_u, c.defocus_u); put3(out->defocus_v, c.defocus_v);
    out->defocus = c.defocus ? 1 : 0;
    out->reserved0 = 0;
}

// getRay(px, py, null): out = origin[3], dir[3], time
void orc_get_ray(const OrcCamera *cam, uint64_t px, uint64_t py, double *out7) {
    const Ray r = toCam(cam).getRay((size_t)px, (size_t)py, nullptr);
    put3(out7, r.origin); put3(out7 + 3, r.dir); out7[6] = r.time;
}

// Tracer.init's height rule, renderer.zig:16,39-40
uint64_t orc_image_height(uint64_t img_w) { return (uint64_t)((double)img_w / (16.0 / 9.0)); }

// ---- scene construction
OrcScene *orc_scene_new() { return new OrcScene(); }
void orc_scene_free(OrcScene *s) { delete s; }

// randomBouncing, rayz.zig:45-168.  The reference draws the scene from the tracer's PRNG
// (rayz.zig:109) seeded from the OS; here the seed is explicit.  Generalisations used by the
// benchmark configs (BASELINE.json configs 4 and 5): the grid loops run a,b in [grid_lo,grid_hi)
// (reference: -11..11), and glass_heavy forces every random sphere and the two non-glass big
// spheres to dielectric (ior 1.5) while consuming the same PRNG draws.
OrcScene *orc_scene_random_bouncing(uint64_t seed, int32_t grid_lo, int32_t grid_hi, int32_t glass_heavy) {
    OrcScene *o = new OrcScene();
    Scene &sc = o->sc;
    Rng rng(seed);
    auto addTex = [&](Texture t) { sc.textures.push_back(t); return (uint32_t)sc.textures.size() - 1; };
    auto addMat = [&](Material m) { sc.materials.push_back(m); return (uint32_t)sc.materials.size() - 1; };
    auto solid = [&](V3 c) { Texture t; t.kind = 1; t.color = c; return t; };
    auto stationary = [&](V3 c, double r, uint32_t m) { Sphere s; s.center.origin = c; s.center.dir = {}; s.radius = r; s.material = m; sc.spheres.push_back(s); };
    // ground :57-73 (innermost struct args first: even, odd, checker, material, sphere)
    {
        V3 even; even.x = 0.2; even.y = 0.3; even.z = 0.1;
        const uint32_t te = addTex(solid(even));
        const uint32_t to = addTex(solid(V3::of(0.9)));
        Texture ck; ck.kind = 0; ck.scale = 0.32; ck.even = te; ck.odd = to;
        const uint32_t tc = addTex(ck);
        Material m; m.kind = 0; m.texture = tc;
        V3 c; c.y = -1000;
        stationary(c, 1000, addMat(m));
    }
    // main three :76-104
    {
        Material m; m.kind = 2; m.ior = 1.5;
        V3 c; c.y = 1;
        stationary(c, 1.0, addMat(m));
    }
    {
        V3 c; c.x = -4; c.y = 1;
        if (glass_heavy) { Material m; m.kind = 2; m.ior = 1.5; stationary(c, 1.0, addMat(m)); }
        else { V3 col; col.x = 0.4; col.y = 0.2; col.z = 0.1; Material m; m.kind = 0; m.texture = addTex(solid(col)); stationary(c, 1.0, addMat(m)); }
    }
    {
        V3 c; c.x = 4; c.y = 1;
        if (glass_heavy) { Material m; m.kind = 2; m.ior = 1.5; stationary(c, 1.0, addMat(m)); }
        else { V3 col; col.x = 0.7; col.y = 0.6; col.z = 0.5; Material m; m.kind = 1; m.fuzz = 0; m.texture = addTex(solid(col)); stationary(c, 1.0, addMat(m)); }
    }
    // randoms :108-166
    for (int a = grid_lo; a < grid_hi; a++) {
        for (int b = grid_lo; b < grid_hi; b++) {
            const double rand_mat = rng.f64();
            V3 center;
            center.x = (double)a + 0.9 * rng.f64();
            center.y = 0.2;
            center.z = (double)b + 0.9 * rng.f64();
            V3 ref; ref.x = 4; ref.y = 0.2; ref.z = 0;
            if (center.sub(ref).mag() <= 0.9) continue;
            Sphere s;
            s.center.origin = center;
            s.center.dir = {};
            s.radius = 0.2;
            if (rand_mat < 0.8) {
                const V3 c1 = rng.v3(0, 1.0);
                const V3 c2 = rng.v3(0, 1.0);
                const double vy = rng.f64() * 0.5;
                if (glass_heavy) { Material m; m.kind = 2; m.ior = 1.5; s.material = addMat(m); }
                else {
                    Material m; m.kind = 0; m.texture = addTex(solid(c1.vmul(c2)));
                    s.material = addMat(m);
                    V3 yh; yh.y = 1;
                    s.center.dir = yh.mul(vy);
                }
            } else if (rand_mat < 0.95) {
                const double fuzz = rng.f64() * 0.5;  // .fuzz evaluated before .texture (:146-149)
                const V3 col = rng.v3(0.5, 1.0);
                if (glass_heavy) { Material m; m.kind = 2; m.ior = 1.5; s.material = addMat(m); }
                else { Material m; m.kind = 1; m.fuzz = fuzz; m.texture = addTex(solid(col)); s.material = addMat(m); }
            } else {
                Material m; m.kind = 2; m.ior = 1.5;
                s.material = addMat(m);
            }
            sc.spheres.push_back(s);
        }
    }
    return o;
}

void orc_scene_counts(const OrcScene *s, uint32_t *ns, uint32_t *nm, uint32_t *nt) {
    *ns = (uint32_t)s->sc.spheres.size(); *nm = (uint32_t)s->sc.materials.size(); *nt = (uint32_t)s->sc.textures.size();
}

void orc_scene_export(const OrcScene *s, double *center, double *velocity, double *radius, uint32_t *sph_mat,
                      uint32_t *mat_kind, double *mat_fuzz, double *mat_ior, uint32_t *mat_tex, uint32_t *mat_method,
                      uint32_t *tex_kind, double *tex_color, double *tex_scale, uint32_t *tex_even, uint32_t *tex_odd) {
    const Scene &sc = s->sc;
    for (size_t i = 0; i < sc.spheres.size(); i++) {
        put3(center + 3 * i, sc.spheres[i].center.origin);
        put3(velocity + 3 * i, sc.spheres[i].center.dir);
        radius[i] = sc.spheres[i].radius;
        sph_mat[i] = sc.spheres[i].material;
    }
    for (size_t i = 0; i < sc.materials.size(); i++) {
        mat_kind[i] = sc.materials[i].kind; mat_fuzz[i] = sc.materials[i].fuzz; mat_ior[i] = sc.materials[i].ior;
        mat_tex[i] = sc.materials[i].texture; mat_method[i] = sc.materials[i].method;
    }
    for (size_t i = 0; i < sc.textures.size(); i++) {
        tex_kind[i] = sc.textures[i].kind; put3(tex_color + 3 * i, sc.textures[i].color);
        tex_scale[i] = sc.textures[i].scale; tex_even[i] = sc.textures[i].even; tex_odd[i] = sc.textures[i].odd;
    }
}

OrcScene *orc_scene_from_arrays(uint32_t ns, uint32_t nm, uint32_t nt, const double *center, const double *velocity,
                                const double *radius, const uint32_t *sph_mat, const uint32_t *mat_kind,
                                const double *mat_fuzz, const double *mat_ior, const uint32_t *mat_tex,
                                const uint32_t *mat_method, const uint32_t *tex_kind, const double *tex_color,
                                const double *tex_scale, const uint32_t *tex_even, const uint32_t *tex_odd) {
    OrcScene *o = new OrcScene();
    Scene &sc = o->sc;
    for (uint32_t i = 0; i < ns; i++) {
        Sphere s;
        s.center.origin = {center[3 * i], center[3 * i + 1], center[3 * i + 2]};
        s.center.dir = {velocity[3 * i], velocity[3 * i + 1], velocity[3 * i + 2]};
        s.radius = radius[i];
        s.material = sph_mat[i];
        sc.spheres.push_back(s);
    }
    for (uint32_t i = 0; i < nm; i++) {
        Material m; m.kind = mat_kind[i]; m.fuzz = mat_fuzz[i]; m.ior = mat_ior[i]; m.texture = mat_tex[i];
        m.method = mat_method ? mat_method[i] : 2;
        sc.materials.push_back(m);
    }
    for (uint32_t i = 0; i < nt; i++) {
        Texture t; t.kind = tex_kind[i]; t.color = {tex_color[3 * i], tex_color[3 * i + 1], tex_color[3 * i + 2]};
        t.scale = tex_scale[i]; t.even = tex_even[i]; t.odd = tex_odd[i];
        sc.textures.push_back(t);
    }
    return o;
}

// ---- the path
// Closest-hit sphere index of getRay(i,j,null) for every pixel; -1 = miss.
void orc_primary_ids(OrcScene *s, const OrcCamera *cam, uint32_t w, uint32_t h, int32_t use_bvh, int32_t *out) {
    Scene &sc = s->sc;
    sc.build();
    const Camera c = toCam(cam);
    for (uint32_t j = 0; j < h; j++)
        for (uint32_t i = 0; i < w; i++) {
            const Ray ray = c.getRay(i, j, nullptr);
            Hit hit;
            const bool have = use_bvh ? sc.findHit(0, ray, 1e-10, INF, hit, nullptr) : sc.findHitBrute(ray, 1e-10, INF, hit);
            out[(size_t)j * w + i] = have ? hit.sphere : -1;
        }
}

// Tracer.render.  threads == 1: the reference's structure exactly — one sequential PRNG
// (seeded with `seed`) over rows x cols x spp.  threads > 1: rows are dealt to std::threads,
// each row with its own PRNG stream Rng(splitmix(seed ^ row)) — a courtesy all-cores mode
// (the reference has no threading, renderer.zig:80-97).  threads == 0 => hardware_concurrency.
// row_streams != 0 forces the per-row streams even with 1 thread (so thread count does not
// change the image).  out_rgb: h*w*3 doubles (linear).  counters (nullable): 10 uint64 in the
// order of RzStats.
uint64_t orc_render(OrcScene *s, const OrcCamera *cam, uint32_t w, uint32_t h, uint32_t spp, uint32_t depth,
                    uint64_t seed, uint32_t threads, int32_t row_streams, int32_t brute, double *out_rgb,
                    uint64_t *counters) {
    Scene &sc = s->sc;
    sc.build();
    const Camera c = toCam(cam);
    Counters total;
    Counters *ct = counters ? &total : nullptr;
    if (threads == 0) threads = std::max(1u, std::thread::hardware_concurrency());
    if (threads == 1 && !row_streams) {
        Rng rng(seed);
        renderRows(sc, c, w, 0, h, spp, depth, rng, brute != 0, out_rgb, ct);
    } else {
        std::atomic<uint32_t> next(0);
        std::vector<Counters> per(threads);
        std::vector<std::thread> pool;
        for (uint32_t t = 0; t < threads; t++)
            pool.emplace_back([&, t]() {
                while (true) {
                    const uint32_t j = next.fetch_add(1);
                    if (j >= h) break;
                    Rng rng(splitmix(seed ^ (0x5851f42d4c957f2dull * (uint64_t)(j + 1))));
                    renderRows(sc, c, w, j, j + 1, spp, depth, rng, brute != 0, out_rgb, counters ? &per[t] : nullptr);
                }
            });
        for (auto &th : pool) th.join();
        for (auto &p : per) total.add(p);
    }
    if (counters) {
        counters[0] = total.paths; counters[1] = total.segments; counters[2] = total.sphere_tests; counters[3] = total.node_tests;
        counters[4] = total.hits[0]; counters[5] = total.hits[1]; counters[6] = total.hits[2];
        counters[7] = total.ended_sky; counters[8] = total.ended_absorbed; counters[9] = total.ended_depth;
    }
    return (uint64_t)w * h * spp;  // renderer.zig:90,100
}

// Image.writePPM's per-pixel transform, image.zig:35-38: sqrt (vec.zig:87-93) -> clamp(0,1) -> trunc(x*255)
void orc_quantise(const double *rgb, uint64_t n_pixels, uint8_t *out) {
    for (uint64_t i = 0; i < n_pixels; i++) {
        V3 px; px.x = rgb[3 * i]; px.y = rgb[3 * i + 1]; px.z = rgb[3 * i + 2];
        const V3 clm = px.sqrt().clamp(0, 1);
        out[3 * i + 0] = (uint8_t)(clm.x * 255);
        out[3 * i + 1] = (uint8_t)(clm.y * 255);
        out[3 * i + 2] = (uint8_t)(clm.z * 255);
    }
}

// ---- small entry points for the reference's known-answer tests
void orc_v3_add(const double *a, const double *b, double *o) { put3(o, V3{a[0], a[1], a[2]}.add({b[0], b[1], b[2]})); }
void orc_v3_mul(const double *a, double v, double *o) { put3(o, V3{a[0], a[1], a[2]}.mul(v)); }
double orc_v3_dot(const double *a, const double *b) { return V3{a[0], a[1], a[2]}.dot({b[0], b[1], b[2]}); }
double orc_v3_mag(const double *a) { return V3{a[0], a[1], a[2]}.mag(); }
void orc_v3_unit(const double *a, double *o) { put3(o, V3{a[0], a[1], a[2]}.unit()); }
int32_t orc_v3_amax(const double *a) { return V3{a[0], a[1], a[2]}.amax(); }
double orc_clamp(double x, double lo, double hi) { return u_clamp(x, lo, hi); }
double orc_min(double a, double b) { return u_min(a, b); }
double orc_max(double a, double b) { return u_max(a, b); }
void orc_refract(const double *unit_dir, const double *norm, double eta, double *o) {
    put3(o, refract({unit_dir[0], unit_dir[1], unit_dir[2]}, {norm[0], norm[1], norm[2]}, eta));
}
double orc_reflectance(double cosv, double ri) { return reflectance(cosv, ri); }
// AABB.init(a,b).hit(ray, tmin, tmax)
int32_t orc_aabb_hit(const double *a, const double *b, const double *origin, const double *dir, double tmin, double tmax) {
    Ray r; r.origin = {origin[0], origin[1], origin[2]}; r.dir = {dir[0], dir[1], dir[2]};
    return AABB::init({a[0], a[1], a[2]}, {b[0], b[1], b[2]}).hit(r, tmin, tmax) ? 1 : 0;
}
// AABB.enclose(AABB.init(a0,a1), AABB.init(b0,b1)) -> low[3], high[3]
void orc_aabb_enclose(const double *a0, const double *a1, const double *b0, const double *b1, double *low, double *high) {
    const AABB r = AABB::enclose(AABB::init({a0[0], a0[1], a0[2]}, {a1[0], a1[1], a1[2]}), AABB::init({b0[0], b0[1], b0[2]}, {b1[0], b1[1], b1[2]}));
    put3(low, r.low); put3(high, r.high);
}
void orc_sphere_bbox(const double *center, const double *velocity, double radius, double *low, double *high) {
    Sphere s; s.center.origin = {center[0], center[1], center[2]}; s.center.dir = {velocity[0], velocity[1], velocity[2]}; s.radius = radius;
    const AABB r = s.boundingBox();
    put3(low, r.low); put3(high, r.high);
}
// Sphere.hitInner: returns 1 + fills t, point[3], normal[3], front_face
int32_t orc_sphere_hit(const double *center, const double *velocity, double radius, const double *origin, const double *dir,
                       double time, double tmin, double tmax, double *out8) {
    Sphere s; s.center.origin = {center[0], center[1], center[2]}; s.center.dir = {velocity[0], velocity[1], velocity[2]}; s.radius = radius;
    Ray r; r.origin = {origin[0], origin[1], origin[2]}; r.dir = {dir[0], dir[1], dir[2]}; r.time = time;
    Hit h;
    if (!s.hit(r, tmin, tmax, h)) return 0;
    out8[0] = h.t; put3(out8 + 1, h.point); put3(out8 + 4, h.normal); out8[7] = h.front_face ? 1 : 0;
    return 1;
}
void orc_texture_value(const OrcScene *s, uint32_t tex, const double *p, double *o) { put3(o, s->sc.textureValue(tex, {p[0], p[1], p[2]})); }
// sky of renderer.zig:124-125 for a direction
void orc_sky(const double *dir, double *o) {
    const double t = 0.5 * (V3{dir[0], dir[1], dir[2]}.unit().y + 1.0);
    V3 blue; blue.x = 0.5; blue.y = 0.7; blue.z = 1.0;
    put3(o, V3::of(1).mul(1.0 - t).add(blue).mul(t));
}
// first n outputs of Rng(seed).f64() — the restated Zig std PRNG
void orc_rng_f64(uint64_t seed, uint32_t n, double *o) { Rng r(seed); for (uint32_t i = 0; i < n; i++) o[i] = r.f64(); }
void orc_rng_u64(uint64_t seed, uint32_t n, uint64_t *o) { Rng r(seed); for (uint32_t i = 0; i < n; i++) o[i] = r.next(); }
// BVH shape export for the device-BVH parity check: per node low[3],high[3] + (left,right,start,end)
uint32_t orc_bvh_export(OrcScene *s, uint32_t max_nodes, double *boxes6, int32_t *links4, uint32_t *order) {
    Scene &sc = s->sc;
    sc.build();
    const uint32_t n = (uint32_t)sc.nodes.size();
    for (uint32_t i = 0; i < n && i < max_nodes; i++) {
        put3(boxes6 + 6 * i, sc.nodes[i].bbox.low); put3(boxes6 + 6 * i + 3, sc.nodes[i].bbox.high);
        links4[4 * i] = sc.nodes[i].left; links4[4 * i + 1] = sc.nodes[i].right;
        links4[4 * i + 2] = (int32_t)sc.nodes[i].starti; links4[4 * i + 3] = (int32_t)sc.nodes[i].endi;
    }
    for (size_t i = 0; i < sc.hittables.size(); i++) order[i] = sc.hittables[i].sphere;
    return n;
}

// ---- path replay (namespace replay above).  The paths of samples [sample_offset, sample_offset + spp) of every pixel of a
// w x h frame, pixel-major (index (j w + i) spp + s).  sampler: 0 Philox, 1 Sobol, 2 Sobol-RQMC.  t_min: the backend's f32
// t_min (0 => 1e-4).  perturb: angle of the perturbed replays (0 => REPLAY_PERTURB).  Outputs per path: rgb[3] clamped radiance, y = its Rec. 709 luminance, segs (closest-hit queries),
// end (0 sky, 1 absorbed, 2 depth), hits[3] per material kind, hash of the event sequence, reason / fseg of the first fragile
// decision (reason 0: robust), tol = the radiance tolerance of a robust path.  threads == 0 => hardware_concurrency.
void orc_replay(OrcScene *s, const OrcCamera *cam, uint32_t w, uint32_t h, uint32_t sample_offset, uint32_t spp, uint32_t depth,
                uint64_t seed, float t_min, int32_t sampler, double perturb, uint32_t threads, double *rgb, double *y, uint32_t *segs, uint8_t *end,
                uint32_t *hits, uint64_t *hash, uint8_t *reason, int32_t *fseg, double *tol) {
    using namespace replay;
    Params P;
    P.sc = &s->sc;
    P.cam = toCam(cam);
    P.depth = depth;
    P.t_min = t_min > 0 ? (double)t_min : (double)1e-4f;   // include/rayz_cuda.h RzRenderParams.t_min
    P.perturb = 0; P.pert_id = 0;
    if (threads == 0) threads = std::max(1u, std::thread::hardware_concurrency());
    std::atomic<uint32_t> next(0);
    auto work = [&]() {
        while (true) {
            const uint32_t j = next.fetch_add(1);
            if (j >= h) break;
            for (uint32_t i = 0; i < w; i++) {
                for (uint32_t sl = 0; sl < spp; sl++) {
                    const size_t q = ((size_t)j * w + i) * spp + sl;
                    const Keys K{(uint32_t)seed, (uint32_t)(seed >> 32), j * w + i, sample_offset + sl, sampler};
                    Path p;
                    trace(K, i, j, P, p);
                    double dev = 0;
                    for (int pr = 0; pr < 2 * REPLAY_PAIRS; pr++) {
                        Params Q = P;
                        Q.perturb = perturb > 0 ? perturb : REPLAY_PERTURB; Q.pert_id = (uint32_t)pr;
                        Path pp;
                        trace(K, i, j, Q, pp);
                        if (pp.ev != p.ev) {
                            size_t e = 0;
                            while (e < p.ev.size() && e < pp.ev.size() && p.ev[e] == pp.ev[e]) e++;
                            fragile(p, R_PERTURB, (uint32_t)e);
                        }
                        for (int c = 0; c < 3; c++) dev = std::fmax(dev, std::fabs(pp.rgb[c] - p.rgb[c]));
                    }
                    uint64_t hh = 0xcbf29ce484222325ull;
                    for (uint64_t e : p.ev) hh = fnv(hh, e);
                    for (int c = 0; c < 3; c++) rgb[3 * q + c] = p.rgb[c];
                    y[q] = 0.2126 * p.rgb[0] + 0.7152 * p.rgb[1] + 0.0722 * p.rgb[2];
                    segs[q] = p.segs;
                    end[q] = (uint8_t)p.end;
                    for (int c = 0; c < 3; c++) hits[3 * q + c] = p.hits[c];
                    hash[q] = hh;
                    reason[q] = (uint8_t)p.reason;
                    fseg[q] = p.fseg;
                    const double mx = std::fmax(p.rgb[0], std::fmax(p.rgb[1], p.rgb[2]));
                    tol[q] = TOL_SAFETY * dev + TOL_REL_PER_SEG * (2.0 * p.segs + 4.0) * mx + TOL_ABS;
                }
            }
        }
    };
    std::vector<std::thread> pool;
    for (uint32_t t = 0; t < threads; t++) pool.emplace_back(work);
    for (auto &t : pool) t.join();
}

// The replay's uniforms of one path: camera ux, uy, ut, ur, ua, then u.x, u.y, u.z, u.w of bounces 1..depth (5 + 4 depth).
void orc_replay_uniforms(uint64_t seed, uint32_t gpix, uint32_t sample, uint32_t depth, int32_t sampler, double *out) {
    const replay::Keys K{(uint32_t)seed, (uint32_t)(seed >> 32), gpix, sample, sampler};
    replay::camera_uniforms(K, out);
    for (uint32_t s = 1; s <= depth; s++) replay::bounce_uniforms(K, s, out + 5 + 4 * (s - 1));
}

}  // extern "C"
