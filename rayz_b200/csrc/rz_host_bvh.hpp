// rz_host_bvh.hpp — host-side tree builders of the C ABI's rayz_cuda_upload_scene (rz_context.cu): the reference-shaped BVH
// K0 walks for the bit-exact primary ids (BVH.build, reference src/hit.zig:130-161) and the binned-SAH BVH2 of the FP32
// traversal kernel K3 for scenes below 8192 spheres (larger ones: rz_bvh_build.cu on the device).  Plain host C++ over
// include/rayz_cuda.h's RzScene and the node records of rz_device.cuh / rz_launch.h; compiled into the library by rz_context.cu and,
// on its own, by tests/hostsim/hostbvh.cu (tree invariants and the rounding helpers on the CPU).  Builds trees only: nothing
// here intersects a ray.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <vector>

#include "../../include/rayz_cuda.h"
#include "rz_device.cuh"
#include "rz_launch.h"   // RzRefNode

namespace {

// min / max that inline to one instruction (no NaNs on this path; std::fmin / std::fmax are libm calls without -ffast-math, and the
// binned SAH build below makes ~600 of them per node: 1.45 ms for the 485-sphere scene, 0.2 ms with these — the same tree)
static inline double dmin(double a, double b) { return b < a ? b : a; }
static inline double dmax(double a, double b) { return b > a ? b : a; }

struct Box {
    double lo[3], hi[3];
    Box() { for (int a = 0; a < 3; a++) { lo[a] = std::numeric_limits<double>::infinity(); hi[a] = -lo[a]; } }
    void grow(const Box &b) { for (int a = 0; a < 3; a++) { lo[a] = dmin(lo[a], b.lo[a]); hi[a] = dmax(hi[a], b.hi[a]); } }
    double area() const {
        const double dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        if (!(dx >= 0) || !(dy >= 0) || !(dz >= 0)) return 0;
        return 2 * (dx * dy + dy * dz + dz * dx);
    }
};

// Sphere.boundingBox (geom.zig:24-31): union of the boxes at center.at(0) and center.at(1)
Box sphere_box(const RzScene &sc, uint32_t i) {
    const double *c = sc.sphere_center + 3 * i, *v = sc.sphere_velocity + 3 * i;
    const double r = sc.sphere_radius[i];
    Box b;
    for (int a = 0; a < 3; a++) {
        const double o1 = c[a], o2 = c[a] + v[a] * 1.0;
        const double l1 = std::fmin(o1 - r, o1 + r), h1 = std::fmax(o1 - r, o1 + r);
        const double l2 = std::fmin(o2 - r, o2 + r), h2 = std::fmax(o2 - r, o2 + r);
        b.lo[a] = std::fmin(l1, l2);
        b.hi[a] = std::fmax(h1, h2);
    }
    return b;
}

// BVH.build (hit.zig:130-161), same shape as the reference: enclose, leaf at <= 2, stable sort
// of the range by bbox.low[longest axis] (amax tie rule vec.zig:150-156), split at n/2.
struct RefBuilder {
    struct H { Box b; uint32_t s; };
    std::vector<H> h;
    std::vector<RzRefNode> nodes;
    int build(size_t si, size_t ei) {
        const int me = (int)nodes.size();
        nodes.push_back(RzRefNode());
        Box bb;
        for (size_t i = si; i < ei; i++) bb.grow(h[i].b);
        for (int a = 0; a < 3; a++) { nodes[me].low[a] = bb.lo[a]; nodes[me].high[a] = bb.hi[a]; }
        nodes[me].left = nodes[me].right = -1;
        nodes[me].start = nodes[me].end = 0;
        const size_t n = ei - si;
        if (n <= 2) {
            nodes[me].start = (int32_t)si;
            nodes[me].end = (int32_t)ei;
        } else {
            const double ex = bb.hi[0] - bb.lo[0], ey = bb.hi[1] - bb.lo[1], ez = bb.hi[2] - bb.lo[2];
            int axis;
            if (ex > ey) axis = ex > ez ? 0 : 2; else axis = ey > ez ? 1 : 2;
            std::stable_sort(h.begin() + si, h.begin() + ei, [axis](const H &a, const H &b) { return a.b.lo[axis] < b.b.lo[axis]; });
            const size_t mid = n / 2 + si;
            const int l = build(si, mid);
            const int r = build(mid, ei);
            nodes[me].left = l;
            nodes[me].right = r;
        }
        return me;
    }
};

// Binned-SAH BVH2 for the FP32 traversal kernel (K3).  Tree shape is ours to choose: closest
// hit does not depend on it.  Leaves hold <= 4 spheres; child boxes are stored in the parent.
struct SahBuilder {
    struct P { Box b; double c[3]; uint32_t s; };
    std::vector<P> p;
    std::vector<RzBvhNode> nodes;
    std::vector<uint32_t> order;  // leaf order of sphere indices
    static constexpr int BINS = 16;
    int LEAF = 4;          // max spheres per leaf (K3 encodes up to 8)
    double node_cost = 0.5; // SAH: cost of one more node visit relative to one sphere test

    // nextafterf(f, -inf) / nextafterf(f, +inf) on the bit pattern (no NaNs here; libm's calls were a third of the build time)
    static float next_down(float f) {
        if (f == -INFINITY) return f;
        if (f == 0.0f) return -std::numeric_limits<float>::denorm_min();
        uint32_t u; memcpy(&u, &f, 4);
        u += f > 0.0f ? 0xffffffffu : 1u;
        memcpy(&f, &u, 4);
        return f;
    }
    static float next_up(float f) { return -next_down(-f); }
    static float down(double v) { float f = (float)v; if ((double)f > v) f = next_down(f); return next_down(f); }
    static float up(double v) { float f = (float)v; if ((double)f < v) f = next_up(f); return next_up(f); }

    struct Ref { int32_t child; uint32_t cnt; Box b; };

    Ref build(size_t si, size_t ei) {
        Box bb, cb;
        for (size_t i = si; i < ei; i++) {
            bb.grow(p[i].b);
            for (int a = 0; a < 3; a++) { cb.lo[a] = dmin(cb.lo[a], p[i].c[a]); cb.hi[a] = dmax(cb.hi[a], p[i].c[a]); }
        }
        const size_t n = ei - si;
        auto make_leaf = [&]() {
            Ref r; r.child = ~(int32_t)order.size(); r.cnt = (uint32_t)n; r.b = bb;
            for (size_t i = si; i < ei; i++) order.push_back(p[i].s);
            return r;
        };
        if (n <= 1) return make_leaf();
        // best binned split over the three axes
        double best_cost = std::numeric_limits<double>::infinity();
        int best_axis = -1, best_bin = -1;
        for (int a = 0; a < 3; a++) {
            const double ext = cb.hi[a] - cb.lo[a];
            if (!(ext > 0)) continue;
            Box bins[BINS]; size_t cnt[BINS] = {0};
            const double k = BINS / ext;
            for (size_t i = si; i < ei; i++) {
                int bi = (int)((p[i].c[a] - cb.lo[a]) * k);
                bi = std::min(std::max(bi, 0), BINS - 1);
                bins[bi].grow(p[i].b); cnt[bi]++;
            }
            double la[BINS], ra[BINS]; size_t lc[BINS], rc[BINS];
            Box acc; size_t c = 0;
            double ar = 0;   // an empty bin changes neither the box nor its area: most bins of the small nodes near the leaves are empty
            for (int i = 0; i < BINS; i++) { if (cnt[i]) { acc.grow(bins[i]); c += cnt[i]; ar = acc.area(); } la[i] = ar; lc[i] = c; }
            acc = Box(); c = 0; ar = 0;
            for (int i = BINS - 1; i >= 0; i--) { if (cnt[i]) { acc.grow(bins[i]); c += cnt[i]; ar = acc.area(); } ra[i] = ar; rc[i] = c; }
            for (int i = 0; i < BINS - 1; i++) {
                if (lc[i] == 0 || rc[i + 1] == 0) continue;
                const double cost = la[i] * (double)lc[i] + ra[i + 1] * (double)rc[i + 1];
                if (cost < best_cost) { best_cost = cost; best_axis = a; best_bin = i; }
            }
        }
        size_t mid;
        if (best_axis < 0) {
            if (n <= (size_t)LEAF) return make_leaf();
            mid = si + n / 2;  // coincident centroids: split by count
        } else {
            const double leaf_cost = bb.area() * (double)n;
            if (n <= (size_t)LEAF && leaf_cost <= best_cost + bb.area() * node_cost) return make_leaf();
            const double ext = cb.hi[best_axis] - cb.lo[best_axis];
            const double k = BINS / ext;
            const double lo = cb.lo[best_axis];
            const int a = best_axis, bbin = best_bin;
            auto it = std::partition(p.begin() + si, p.begin() + ei, [&](const P &q) {
                int bi = (int)((q.c[a] - lo) * k);
                bi = std::min(std::max(bi, 0), BINS - 1);
                return bi <= bbin;
            });
            mid = (size_t)(it - p.begin());
            if (mid == si || mid == ei) mid = si + n / 2;
        }
        const int me = (int)nodes.size();
        nodes.push_back(RzBvhNode());
        const Ref l = build(si, mid);
        const Ref r = build(mid, ei);
        set_child(me, 0, l);
        set_child(me, 1, r);
        Ref out; out.child = me; out.cnt = 0; out.b = bb;
        return out;
    }
    void set_child(int node, int c, const Ref &r) {
        RzBvhNode &n = nodes[node];
        n.lox[c] = down(r.b.lo[0]); n.hix[c] = up(r.b.hi[0]);
        n.loy[c] = down(r.b.lo[1]); n.hiy[c] = up(r.b.hi[1]);
        n.loz[c] = down(r.b.lo[2]); n.hiz[c] = up(r.b.hi[2]);
        n.child[c] = r.child; n.cnt[c] = r.cnt;
    }
    void run() {
        nodes.clear(); order.clear();
        if (p.empty()) { nodes.push_back(empty_node()); return; }
        const Ref root = build(0, p.size());
        if (root.child < 0) {  // whole scene is one leaf: wrap it
            nodes.clear();
            nodes.push_back(empty_node());
            set_child(0, 0, root);
        }
        // build() creates parents before children and the root first => node 0 is the root
    }
    static RzBvhNode empty_node() {
        RzBvhNode n;
        for (int c = 0; c < 2; c++) {
            n.lox[c] = n.loy[c] = n.loz[c] = INFINITY;
            n.hix[c] = n.hiy[c] = n.hiz[c] = -INFINITY;
            n.child[c] = ~0; n.cnt[c] = 0;
        }
        return n;
    }
};

}  // namespace
