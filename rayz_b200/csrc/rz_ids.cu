// rz_ids.cu — K0: f64, FMA-free closest-hit sphere index of the deterministic primary ray.
//
// COMPILED WITH --fmad=false: the reference's float mode is strict (Zig never fuses a*b+c),
// f64 division and sqrt are IEEE-correct on both sides, so every intermediate below is bit
// identical to the reference's arithmetic and the ids are exact, not "close".
//
// Restates, operation for operation (paths under /root/reference/src):
//   Camera.getRay(px, py, null)   camera.zig:59-77   (pixel centre, no defocus, time 0)
//   AABB.hit                      hit.zig:70-98      (true divides, strict t1 > t0)
//   BVH.findHit                   hit.zig:181-216    (left before right, tmax := closest so far)
//   Sphere.hitInner               geom.zig:38-66     (closed [tmin,tmax] root acceptance)
// The recursion of findHit is an explicit stack here: every accepted hit has t <= the tmax in
// force, so "tmax passed down" always equals the running closest t and a depth-first,
// left-first walk with one running `best` visits and accepts exactly what the recursion does.
#include "rz_launch.h"   // RzRefNode, RzIdsArgs

struct D3 { double x, y, z; };
__device__ __forceinline__ D3 d3(double x, double y, double z) { D3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ D3 add(D3 a, D3 b) { return d3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ D3 sub(D3 a, D3 b) { return d3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ D3 mul(D3 a, double v) { return d3(a.x * v, a.y * v, a.z * v); }
__device__ __forceinline__ double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }  // (x*x + y*y) + z*z

// Sphere.hitInner; only t matters for the id (point/normal are not needed to pick the sphere)
__device__ __forceinline__ bool sphere_hit(const double4 c, const double4 v, D3 ro, D3 rd, double time, double tmin,
                                           double tmax, double &t_out) {
    const D3 origin_now = add(d3(c.x, c.y, c.z), mul(d3(v.x, v.y, v.z), time));
    const D3 offset = sub(origin_now, ro);
    const double a = dot(rd, rd);
    const double half_b = dot(rd, offset);
    const double cc = dot(offset, offset) - c.w * c.w;
    const double discriminant = half_b * half_b - a * cc;
    if (discriminant < 0) return false;
    const double rt = sqrt(discriminant);
    const double t1 = (half_b - rt) / a;
    const double t2 = (half_b + rt) / a;
    if (t1 >= tmin && t1 <= tmax) { t_out = t1; return true; }
    if (t2 >= tmin && t2 <= tmax) { t_out = t2; return true; }
    return false;
}

__device__ __forceinline__ bool aabb_hit(const RzRefNode &n, D3 ro, D3 rd, double tmin, double tmax) {
    const double t0s[3] = {(n.low[0] - ro.x) / rd.x, (n.low[1] - ro.y) / rd.y, (n.low[2] - ro.z) / rd.z};
    const double t1s[3] = {(n.high[0] - ro.x) / rd.x, (n.high[1] - ro.y) / rd.y, (n.high[2] - ro.z) / rd.z};
    double t0 = tmin, t1 = tmax;
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {
        const double v0 = t0s[ax], v1 = t1s[ax];
        if (v0 < v1) {
            t0 = fmax(v0, t0);  // @max/@min: NaN operand ignored, like fmax/fmin
            t1 = fmin(v1, t1);
        } else {
            t0 = fmax(v1, t0);
            t1 = fmin(v0, t1);
        }
    }
    return t1 > t0;
}

__global__ void __launch_bounds__(128) rz_ids_kernel(const RzIdsArgs a) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.width * a.height) return;
    const uint32_t py = idx / a.width, px = idx - py * a.width;
    // getRay(px, py, null): dir = px_du*x + px_dv*y + px_origin - origin
    const double x = (double)px, y = (double)py;
    const D3 ro = d3(a.look_from[0], a.look_from[1], a.look_from[2]);
    const D3 rd = sub(add(add(mul(d3(a.px_du[0], a.px_du[1], a.px_du[2]), x), mul(d3(a.px_dv[0], a.px_dv[1], a.px_dv[2]), y)),
                          d3(a.px_origin[0], a.px_origin[1], a.px_origin[2])),
                      ro);
    const double tmin = 1e-10;                       // renderer.zig:107
    double best = __longlong_as_double(0x7ff0000000000000ll);  // +inf
    int32_t id = -1;
    if (!a.use_bvh) {
        for (uint32_t i = 0; i < a.n_spheres; i++) {
            double t;
            if (sphere_hit(a.c64[i], a.v64[i], ro, rd, 0.0, tmin, best, t)) { best = t; id = (int32_t)i; }
        }
    } else if (a.n_nodes > 0) {
        int32_t stack[64];
        int sp = 0;
        stack[sp++] = 0;
        while (sp > 0) {
            const RzRefNode &n = a.nodes[stack[--sp]];
            if (!aabb_hit(n, ro, rd, tmin, best)) continue;
            if (n.left >= 0) {
                if (sp < 63) { stack[sp++] = n.right; stack[sp++] = n.left; }
                else atomicOr(a.err, 2u);   // the reference-shaped tree is balanced (depth <= log2 n + 1): cannot happen below 2^60 spheres
                continue;
            }
            for (int32_t i = n.start; i < n.end; i++) {
                const uint32_t s = a.order[i];
                double t;
                if (sphere_hit(a.c64[s], a.v64[s], ro, rd, 0.0, tmin, best, t)) { best = t; id = (int32_t)s; }
            }
        }
    }
    a.out[idx] = id;
}

extern "C" cudaError_t rz_launch_ids(const RzIdsArgs *a, cudaStream_t stream) {
    const uint32_t n = a->width * a->height;
    rz_ids_kernel<<<(n + 127) / 128, 128, 0, stream>>>(*a);
    return cudaGetLastError();
}
