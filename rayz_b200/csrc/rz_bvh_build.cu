// rz_bvh_build.cu — K4: device-side BVH build (LBVH) for the FP32 traversal kernel K3.
//
// Replaces, for large scenes, the role of BVH.build (reference src/hit.zig:130-161, driven from
// Tracer.render renderer.zig:76-78) + Sphere.boundingBox (geom.zig:24-31).  The reference sorts the
// range at every level (O(N log^2 N), recursive, pointer-linked nodes); the closest-hit result does
// not depend on the tree shape, so the device build is free to use a different construction:
//
//   1. boxes     : per sphere, the union of its boxes at time 0 and 1 (geom.zig:24-31) in f64,
//                  rounded OUTWARD to f32 and padded by one more ulp (like the host SAH builder);
//                  scene-wide centroid bounds by warp reduction + ordered-int atomics
//   2. morton    : 63-bit Morton code of the box centroid (21 bits per axis)
//   3. sort      : cub::DeviceRadixSort::SortPairs (key = code, value = sphere index)  [library]
//   4. hierarchy : Karras 2012 ("Maximizing parallelism in the construction of BVHs, octrees and
//                  k-d trees"): internal node i covers a key range found by binary search on the
//                  common-prefix length; ties between equal codes are broken by the index
//   5. refit     : bottom-up, one thread per leaf, an atomic arrival counter per internal node; the
//                  second arriver unions the two child boxes and continues upwards
//   6. emit      : RzBvhNode records of K3 (both child boxes in the parent); subtrees of <= leaf_max
//                  spheres collapse into one leaf (their leaves are contiguous in sorted order) —
//                  leaf_max = RzTuning::lbvh_leaf, default 1: a 4-sphere leaf saves 6 of 53 box tests
//                  per ray segment and costs 5 more sphere tests, each divergent (config 4: 1735 vs
//                  1872 Mpaths/s); the sphere set is gathered into leaf order
//
// One launch sequence on the caller's stream, no host round trip except the sort's temp-size query.
#include <cub/device/device_radix_sort.cuh>

#include "rz_device.cuh"
#include "rz_launch.h"

namespace {


struct LbvhTemp {
    float *lo, *hi;                 // [n][3] padded f32 sphere boxes
    unsigned long long *keys_in, *keys_out;
    uint32_t *vals_in, *vals_out;   // vals_out = leaf order
    int *left, *right, *parent;     // internal nodes [n-1]; child >= 0 internal, < 0 => ~leaf
    int *leaf_parent;               // [n]
    int *first, *last;              // key range of each internal node
    float *nlo, *nhi;               // [n-1][3] internal node boxes
    unsigned int *arrive;           // [n-1]
    int *bounds;                    // 6 ordered ints: centroid lo xyz, hi xyz
};

__device__ __forceinline__ int f2ord(float f) { const int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }
__device__ __forceinline__ float rz_down(double v) { return nextafterf(__double2float_rd(v), -INFINITY); }
__device__ __forceinline__ float rz_up(double v) { return nextafterf(__double2float_ru(v), INFINITY); }

__global__ void lbvh_init_bounds(int *bounds) {
    if (threadIdx.x < 3) bounds[threadIdx.x] = 0x7fffffff;
    else if (threadIdx.x < 6) bounds[threadIdx.x] = (int)0x80000000;
}

// 1. boxes + centroid bounds
__global__ void __launch_bounds__(256) lbvh_boxes(const double4 *c64, const double4 *v64, uint32_t n, LbvhTemp t) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    float c[3] = {0.f, 0.f, 0.f};
    const bool live = i < n;
    if (live) {
        const double4 cc = c64[i], vv = v64[i];
        const double ce[3] = {cc.x, cc.y, cc.z}, ve[3] = {vv.x, vv.y, vv.z}, r = cc.w;
#pragma unroll
        for (int a = 0; a < 3; a++) {
            const double o2 = ce[a] + ve[a] * 1.0;                               // center.at(1), geom.zig:27
            const double lo = fmin(ce[a] - r, o2 - r), hi = fmax(ce[a] + r, o2 + r);
            const float flo = rz_down(lo), fhi = rz_up(hi);
            t.lo[3 * i + a] = flo;
            t.hi[3 * i + a] = fhi;
            c[a] = 0.5f * (flo + fhi);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; a++) {
        int lo = live ? f2ord(c[a]) : 0x7fffffff, hi = live ? f2ord(c[a]) : (int)0x80000000;
        for (int o = 16; o > 0; o >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if ((threadIdx.x & 31) == 0) { atomicMin(t.bounds + a, lo); atomicMax(t.bounds + 3 + a, hi); }
    }
}

__device__ __forceinline__ unsigned long long expand21(unsigned long long v) {   // spread 21 bits to every third bit
    v &= 0x1fffffull;
    v = (v | v << 32) & 0x1f00000000ffffull;
    v = (v | v << 16) & 0x1f0000ff0000ffull;
    v = (v | v << 8) & 0x100f00f00f00f00full;
    v = (v | v << 4) & 0x10c30c30c30c30c3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
}

// 2. Morton codes
__global__ void __launch_bounds__(256) lbvh_morton(uint32_t n, LbvhTemp t) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned long long code = 0;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        const float lo = ord2f(t.bounds[a]), hi = ord2f(t.bounds[3 + a]);
        const float c = 0.5f * (t.lo[3 * i + a] + t.hi[3 * i + a]);
        const float ext = hi - lo;
        float u = ext > 0.f ? (c - lo) / ext : 0.f;
        u = fminf(fmaxf(u, 0.f), 1.f);
        const unsigned long long q = (unsigned long long)fminf(u * 2097152.f, 2097151.f);
        code |= expand21(q) << (2 - a);
    }
    t.keys_in[i] = code;
    t.vals_in[i] = i;
}

// common-prefix length of keys i and j (Karras): equal codes fall back to the index bits
__device__ __forceinline__ int lbvh_delta(const unsigned long long *keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    const unsigned long long a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz((unsigned)i ^ (unsigned)j);
    return __clzll((long long)(a ^ b));
}

// 4. hierarchy: internal node i in [0, n-1)
__global__ void __launch_bounds__(256) lbvh_hierarchy(uint32_t n, LbvhTemp t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = (int)n;
    if (i >= N - 1) return;
    const unsigned long long *keys = t.keys_out;
    const int d = lbvh_delta(keys, N, i, i + 1) > lbvh_delta(keys, N, i, i - 1) ? 1 : -1;
    const int dmin = lbvh_delta(keys, N, i, i - d);
    int lmax = 2;
    while (lbvh_delta(keys, N, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int s = lmax >> 1; s >= 1; s >>= 1)
        if (lbvh_delta(keys, N, i, i + (l + s) * d) > dmin) l += s;
    const int j = i + l * d;
    const int dnode = lbvh_delta(keys, N, i, j);
    int s = 0;
    int step = l;
    do {
        step = (step + 1) >> 1;
        if (lbvh_delta(keys, N, i, i + (s + step) * d) > dnode) s += step;
    } while (step > 1);
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int lc = (lo == gamma) ? ~gamma : gamma;            // leaf if the left part is one key
    const int rc = (hi == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    t.left[i] = lc;
    t.right[i] = rc;
    t.first[i] = lo;
    t.last[i] = hi;
    if (lc >= 0) t.parent[lc] = i; else t.leaf_parent[~lc] = i;
    if (rc >= 0) t.parent[rc] = i; else t.leaf_parent[~rc] = i;
    if (i == 0) t.parent[0] = -1;
    t.arrive[i] = 0u;
}

// 5. refit
__global__ void __launch_bounds__(256) lbvh_refit(uint32_t n, LbvhTemp t) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;   // leaf position in sorted order
    if (k >= n) return;
    int node = t.leaf_parent[k];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(t.arrive + node, 1u) == 0u) return;       // first arriver: the sibling is not ready yet
        float lo[3], hi[3];
#pragma unroll
        for (int a = 0; a < 3; a++) { lo[a] = INFINITY; hi[a] = -INFINITY; }
        const int ch[2] = {t.left[node], t.right[node]};
#pragma unroll
        for (int c = 0; c < 2; c++) {
            const float *plo, *phi;
            if (ch[c] < 0) { const uint32_t s = t.vals_out[~ch[c]]; plo = t.lo + 3 * s; phi = t.hi + 3 * s; }
            else { plo = t.nlo + 3 * ch[c]; phi = t.nhi + 3 * ch[c]; }
#pragma unroll
            for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], __ldcg(plo + a)); hi[a] = fmaxf(hi[a], __ldcg(phi + a)); }
        }
#pragma unroll
        for (int a = 0; a < 3; a++) { __stcg(t.nlo + 3 * node + a, lo[a]); __stcg(t.nhi + 3 * node + a, hi[a]); }
        node = t.parent[node];
    }
}

// 6a. K3 node records.  One thread per internal node; nodes inside a collapsed subtree are never
// referenced and are left as empty records.
__global__ void __launch_bounds__(256) lbvh_emit(uint32_t n, LbvhTemp t, RzBvhNode *out, int leaf_max) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = (int)n;
    if (i >= max(N - 1, 1)) return;
    RzBvhNode nd;
#pragma unroll
    for (int c = 0; c < 2; c++) {
        nd.lox[c] = nd.loy[c] = nd.loz[c] = INFINITY;
        nd.hix[c] = nd.hiy[c] = nd.hiz[c] = -INFINITY;
        nd.child[c] = ~0; nd.cnt[c] = 0u;
    }
    if (N == 1) {   // one sphere: a root with a single leaf child
        const uint32_t s = t.vals_out[0];
        nd.lox[0] = t.lo[3 * s]; nd.loy[0] = t.lo[3 * s + 1]; nd.loz[0] = t.lo[3 * s + 2];
        nd.hix[0] = t.hi[3 * s]; nd.hiy[0] = t.hi[3 * s + 1]; nd.hiz[0] = t.hi[3 * s + 2];
        nd.child[0] = ~0; nd.cnt[0] = 1u;
        out[0] = nd;
        return;
    }
    const int ch[2] = {t.left[i], t.right[i]};
#pragma unroll
    for (int c = 0; c < 2; c++) {
        const float *plo, *phi;
        int child;
        uint32_t cnt;
        if (ch[c] < 0) {
            const uint32_t s = t.vals_out[~ch[c]];
            plo = t.lo + 3 * s; phi = t.hi + 3 * s;
            child = ch[c]; cnt = 1u;
        } else {
            plo = t.nlo + 3 * ch[c]; phi = t.nhi + 3 * ch[c];
            const int count = t.last[ch[c]] - t.first[ch[c]] + 1;
            if (count <= leaf_max) { child = ~t.first[ch[c]]; cnt = (uint32_t)count; }   // collapse the subtree
            else { child = ch[c]; cnt = 0u; }
        }
        nd.child[c] = child; nd.cnt[c] = cnt;
        if (c == 0) { nd.lox[0] = plo[0]; nd.loy[0] = plo[1]; nd.loz[0] = plo[2]; nd.hix[0] = phi[0]; nd.hiy[0] = phi[1]; nd.hiz[0] = phi[2]; }
        else { nd.lox[1] = plo[0]; nd.loy[1] = plo[1]; nd.loz[1] = plo[2]; nd.hix[1] = phi[0]; nd.hiy[1] = phi[1]; nd.hiz[1] = phi[2]; }
    }
    out[i] = nd;
}

// 6b. sphere set in leaf order (the SoA operands of K3, layout of RzSphereSet)
__global__ void __launch_bounds__(256) lbvh_gather_set(uint32_t n, const uint32_t *order, const double4 *c64, const double4 *v64,
                                                      const uint32_t *mat, float4 *o_cr, float4 *o_vel, double4 *o_c64,
                                                      double4 *o_v64, uint32_t *o_mat, int32_t *o_orig) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t s = order[k];
    const double4 c = c64[s], v = v64[s];
    o_cr[k] = make_float4((float)c.x, (float)c.y, (float)c.z, -(float)(c.w * c.w));
    o_vel[k] = make_float4((float)v.x, (float)v.y, (float)v.z, (float)c.w);
    o_c64[k] = c;
    o_v64[k] = make_double4(v.x, v.y, v.z, 1.0 / c.w);   // .w = 1 / radius for rz_refine_hit
    o_mat[k] = mat[s];
    o_orig[k] = (int32_t)s;
}

// 7. finalize (both builders' trees): leaves get the reference the traversal follows (rz_leaf_ref), and an unused slot — only
//    the root of a scene that is one leaf has one — becomes a copy of its sibling (visited twice at worst: the second visit
//    finds nothing nearer), so that K3's node visit is slab tests and nothing else.
__global__ void __launch_bounds__(256) bvh_finalize(RzBvhNode *nodes, uint32_t n_nodes) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    RzBvhNode nd = nodes[i];
    bool empty[2];
#pragma unroll
    for (int c = 0; c < 2; c++) {
        empty[c] = nd.child[c] < 0 && nd.cnt[c] == 0u;
        if (nd.child[c] < 0 && nd.cnt[c] != 0u) nd.child[c] = rz_leaf_ref(nd.child[c], nd.cnt[c]);
    }
#pragma unroll
    for (int c = 0; c < 2; c++) {
        if (empty[c] && !empty[1 - c]) {
            const int o = 1 - c;
            nd.lox[c] = nd.lox[o]; nd.hix[c] = nd.hix[o]; nd.loy[c] = nd.loy[o]; nd.hiy[c] = nd.hiy[o]; nd.loz[c] = nd.loz[o]; nd.hiz[c] = nd.hiz[o];
            nd.child[c] = nd.child[o]; nd.cnt[c] = nd.cnt[o];
        }
    }
    nodes[i] = nd;
}

}  // namespace

// Turns a freshly built tree (either builder's) into the form K3 traverses.  Once per tree: applying it twice would encode twice.
extern "C" cudaError_t rz_bvh_finalize(RzBvhNode *nodes, uint32_t n_nodes, cudaStream_t stream) {
    if (n_nodes == 0) return cudaSuccess;
    bvh_finalize<<<(n_nodes + 255u) / 256u, 256, 0, stream>>>(nodes, n_nodes);
    return cudaGetLastError();
}

// Bytes of scratch the build needs for n spheres (the caller allocates once and may reuse it).
extern "C" size_t rz_lbvh_scratch_bytes(uint32_t n) {
    size_t sort_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)n, 0, 63);
    const size_t N = n ? n : 1;
    size_t b = 0;
    b += 2 * (3 * N * sizeof(float));            // lo, hi
    b += 2 * (N * sizeof(unsigned long long));   // keys
    b += 2 * (N * sizeof(uint32_t));             // vals
    b += 6 * (N * sizeof(int));                  // left right parent leaf_parent first last
    b += 2 * (3 * N * sizeof(float));            // nlo nhi
    b += N * sizeof(unsigned int);               // arrive
    b += 64;                                     // bounds
    b += sort_bytes + 256 * 16;                  // sort temp + alignment slack
    return b;
}

// Builds the K3 tree on `stream`.  Inputs: the scene's f64 spheres in caller order (c64: xyz + radius,
// v64: velocity), material index per sphere.  Outputs: `nodes` (max(n-1,1) records, root = 0) and the
// leaf-ordered sphere set arrays (n entries each).  Everything is device memory.
extern "C" cudaError_t rz_lbvh_build(uint32_t n, int leaf_max, const double4 *c64, const double4 *v64, const uint32_t *mat, void *scratch,
                                     size_t scratch_bytes, RzBvhNode *nodes, float4 *o_cr, float4 *o_vel, double4 *o_c64,
                                     double4 *o_v64, uint32_t *o_mat, int32_t *o_orig, cudaStream_t stream) {
    if (n == 0) return cudaErrorInvalidValue;
    if (scratch_bytes < rz_lbvh_scratch_bytes(n)) return cudaErrorInvalidValue;
    const size_t N = n;
    unsigned char *p = static_cast<unsigned char *>(scratch);
    auto take = [&](size_t bytes) { void *q = p; p += (bytes + 255) & ~size_t(255); return q; };
    LbvhTemp t;
    t.lo = (float *)take(3 * N * 4); t.hi = (float *)take(3 * N * 4);
    t.keys_in = (unsigned long long *)take(N * 8); t.keys_out = (unsigned long long *)take(N * 8);
    t.vals_in = (uint32_t *)take(N * 4); t.vals_out = (uint32_t *)take(N * 4);
    t.left = (int *)take(N * 4); t.right = (int *)take(N * 4); t.parent = (int *)take(N * 4);
    t.leaf_parent = (int *)take(N * 4); t.first = (int *)take(N * 4); t.last = (int *)take(N * 4);
    t.nlo = (float *)take(3 * N * 4); t.nhi = (float *)take(3 * N * 4);
    t.arrive = (unsigned int *)take(N * 4);
    t.bounds = (int *)take(64);
    void *sort_tmp = p;
    size_t sort_bytes = scratch_bytes - (size_t)(p - static_cast<unsigned char *>(scratch));

    const unsigned grid = (unsigned)((N + 255) / 256);
    lbvh_init_bounds<<<1, 32, 0, stream>>>(t.bounds);
    lbvh_boxes<<<grid, 256, 0, stream>>>(c64, v64, n, t);
    lbvh_morton<<<grid, 256, 0, stream>>>(n, t);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, t.keys_in, t.keys_out, t.vals_in, t.vals_out, (int)n, 0, 63, stream);
    if (e != cudaSuccess) return e;
    if (n > 1) {
        lbvh_hierarchy<<<grid, 256, 0, stream>>>(n, t);
        lbvh_refit<<<grid, 256, 0, stream>>>(n, t);
    }
    lbvh_emit<<<grid, 256, 0, stream>>>(n, t, nodes, leaf_max);
    lbvh_gather_set<<<grid, 256, 0, stream>>>(n, t.vals_out, c64, v64, mat, o_cr, o_vel, o_c64, o_v64, o_mat, o_orig);
    return cudaGetLastError();
}
