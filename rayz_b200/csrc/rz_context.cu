// rz_context.cu — host side of the C ABI (include/rayz_cuda.h): contexts, scene flattening,
// BVH builds, kernel orchestration, peer gather.  No CPU rendering path exists here: every
// entry point that produces pixels or ids launches CUDA kernels or fails.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rayz_cuda.h"
#include "rz_device.cuh"
#include "rz_host_bvh.hpp"   // Box, sphere_box, RefBuilder (K0's reference-shaped BVH), SahBuilder (K3's tree for small scenes); RzRefNode

// from rz_path.cu / rz_ids.cu / rz_misc.cu / rz_wavefront.cu
struct RzIdsArgs {
    const RzRefNode *nodes; const uint32_t *order; const double4 *c64; const double4 *v64;
    uint32_t n_spheres, n_nodes; double look_from[3], px_du[3], px_dv[3], px_origin[3];
    uint32_t width, height; int use_bvh; int32_t *out; unsigned int *err;
};
struct RzResolveArgs {
    const unsigned long long *accum; float4 *out_linear; uint8_t *out_rgb8; float *out_err;
    uint32_t n_local_px, width; uint32_t spp; uint32_t dev_index, dev_count, band_rows;
};
extern "C" cudaError_t rz_launch_path(const RzPathArgs *a, int rays_per_thread, int collect_stats, int sm_count,
                                      cudaStream_t stream, int *grid_out);
extern "C" cudaError_t rz_path_warm(void);
extern "C" size_t rz_primary_smem_bytes(const RzPathArgs *a);
extern "C" cudaError_t rz_launch_second(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream);
extern "C" size_t rz_bin_scratch_bytes(void);
extern "C" cudaError_t rz_launch_bin_lists(const RzPathArgs *a, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_second_grid(const RzPathArgs *a, int collect_stats, int sm_count, int *grid);
extern "C" cudaError_t rz_bin_sort(const unsigned short *keys_in, const unsigned int *count, uint32_t cap, unsigned int *bins,
                                   unsigned short *keys_out, uint32_t *idx_out, uint32_t ue_max, uint32_t ue_div, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_sort_warm(void);
extern "C" cudaError_t rz_launch_primary(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_bvh_warm(void);
extern "C" uint32_t rz_bvh_camera_tile_w(void);
extern "C" cudaError_t rz_launch_bvh(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream);
extern "C" cudaError_t rz_launch_bvh_stage(const RzPathArgs *a, int collect_stats, int sm_count, cudaStream_t stream);
extern "C" size_t rz_lbvh_scratch_bytes(uint32_t n);
extern "C" cudaError_t rz_bvh_finalize(RzBvhNode *nodes, uint32_t n_nodes, cudaStream_t stream);
extern "C" cudaError_t rz_lbvh_build(uint32_t n, int leaf_max, const double4 *c64, const double4 *v64, const uint32_t *mat, void *scratch,
                                     size_t scratch_bytes, RzBvhNode *nodes, float4 *o_cr, float4 *o_vel, double4 *o_c64,
                                     double4 *o_v64, uint32_t *o_mat, int32_t *o_orig, cudaStream_t stream);
extern "C" size_t rz_bvh_wide_scratch_bytes(uint32_t n_nodes);
extern "C" cudaError_t rz_bvh_wide_collapse(const RzBvhNode *n2, uint32_t n_nodes, void *scratch, RzBvh4Node *out, cudaStream_t stream);
extern "C" cudaError_t rz_launch_ids(const RzIdsArgs *a, cudaStream_t stream);
extern "C" cudaError_t rz_launch_resolve(const RzResolveArgs *a, cudaStream_t stream);
extern "C" uint32_t rz_noise_grid(void);
extern "C" cudaError_t rz_launch_noise_reduce(const unsigned long long *accum, uint32_t n_local_px, uint32_t n, double target, void *out,
                                              cudaStream_t stream);
extern "C" cudaError_t rz_launch_ffma_peak(float *sink, int grid, int iters, int mode, cudaStream_t stream);
extern "C" cudaError_t rz_wavefront_render(const RzPathArgs *a, int sm_count, int collect_stats, cudaStream_t stream,
                                           void **scratch, size_t *scratch_bytes, uint32_t *launches);
extern "C" void rz_wavefront_free(void *scratch);

// ------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
static int rz_fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
#define RZ_CUDA(call)                                                                                   \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return rz_fail(e_ == cudaErrorMemoryAllocation ? RZ_ERR_OOM : RZ_ERR_CUDA, "%s:%d %s -> %s", \
                           __FILE__, __LINE__, #call, cudaGetErrorString(e_));                          \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    DeviceGuard() { cudaGetDevice(&prev); }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ------------------------------------------------------------------------------ device state
template <class T>
struct DBuf {
    T *p = nullptr;
    size_t n = 0;
    int alloc(size_t count) {
        if (count <= n && p) return RZ_OK;
        release();
        if (count == 0) count = 1;
        RZ_CUDA(cudaMalloc((void **)&p, count * sizeof(T)));
        n = count;
        return RZ_OK;
    }
    int upload(const std::vector<T> &h, cudaStream_t s) {
        int rc = alloc(h.size());
        if (rc) return rc;
        if (!h.empty()) RZ_CUDA(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s));
        return RZ_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

struct SetBufs {
    DBuf<float4> cr, vel, pk;
    DBuf<double4> c64, v64;
    DBuf<uint32_t> mat;
    DBuf<int32_t> orig;
    uint32_t n = 0, n_static = 0, n_static_pad = 0, n_pad = 0;
    RzSphereSet view() const {
        RzSphereSet s;
        s.cr = cr.p; s.vel = vel.p; s.pk = pk.p; s.c64 = c64.p; s.v64 = v64.p; s.mat = mat.p; s.orig = orig.p;
        s.n = n; s.n_static = n_static; s.n_static_pad = n_static_pad; s.n_pad = n_pad;
        return s;
    }
    void release() { cr.release(); vel.release(); pk.release(); c64.release(); v64.release(); mat.release(); orig.release(); }
};

struct Dev {
    int id = 0, sms = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t stream2 = nullptr;   // staged K1: odd passes run here so that a pass fills the tail of the previous one
    cudaEvent_t ev_s2 = nullptr, ev_tab = nullptr;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // start, path0, path1, resolve1, done
    SetBufs brute, bvhset;
    DBuf<RzBvhNode> bvh;              // the builders' binary tree (host SAH or device LBVH): input of the collapse
    DBuf<RzBvh4Node> bvh4;            // what K3 walks: every second level collapsed (rz_bvh_wide.cu)
    DBuf<int> wide_scratch;
    uint32_t bvh_nodes = 0;
    DBuf<int32_t> brute_to_bvh;       // staged K1 with a BVH tail: position in `brute` -> position in `bvhset` (empty: no such tail)
    DBuf<RzRefNode> refnodes;
    DBuf<uint32_t> reforder;
    DBuf<double4> c64_orig, v64_orig;
    DBuf<uint32_t> mat_orig;
    DBuf<unsigned char> lbvh_scratch;
    uint32_t n_refnodes = 0;
    DBuf<uint32_t> m_kind, m_tex, m_method, t_kind, t_even, t_odd;
    DBuf<float> m_fuzz, m_ior;
    DBuf<float4> m_rec;
    DBuf<float4> t_color;
    DBuf<double> t_inv_scale;
    DBuf<unsigned long long> accum;
    // staged K1, one set per side (passes alternate between two streams): q1 = after the camera segment, q2 = after the second
    DBuf<float4> q1[2], q2[2];
    DBuf<unsigned short> keys[2];
    DBuf<uint32_t> idx_sorted[2];
    DBuf<unsigned int> bins[2];       // rz_sort.cu: per-key counts / cursors of the side's sort (RZ_BIN_* layout)
    DBuf<unsigned char> bin_lists;    // per sort group: the reachable sphere pairs in reach-class order (rz_bin_lists_kernel)
    DBuf<unsigned int> counter;
    DBuf<unsigned int> errword;       // device error word (RZ_DEV_ERR_*), cleared at the start of every render / ids call
    DBuf<RzStatsDev> stats;
    DBuf<float4> out_linear;
    DBuf<uint8_t> out_rgb8;
    DBuf<float> out_err;              // rayz_cuda_noise: per-pixel error of the context's rows (gather root only)
    DBuf<double> noise_part;          // rayz_cuda_noise: the reduction's per-CTA partials of this device
    DBuf<float4> loc_linear;          // multi-device render into HOST buffers: this device's own rows, copied out over its own PCIe link
    DBuf<uint8_t> loc_rgb8;
    uint32_t loc_rows = 0;            // rows of the last such render
    DBuf<int32_t> ids;
    DBuf<float> sink;
    void *wf_scratch = nullptr;
    size_t wf_scratch_bytes = 0;
    std::vector<cudaEvent_t> pass_ev;   // staged K1: [3i] after the primary kernel of pass i, [3i+1] after the sorted stages, [3i+2] after the tail kernel
    std::vector<cudaEvent_t> stage_ev;  // staged K1: per pass and sorted stage, [2k] after the sort, [2k+1] after the kernel
    uint32_t n_second = 0;              // sorted stages per pass of the last render
    uint32_t queue_entries = 0;         // entries per queue buffer of the last render (0 = not the staged form)
    uint32_t passes = 0;                // passes of the last render (0 = not the staged form)
    bool serial_passes = false;
};

// What the accumulators of the context's devices hold (RZ_RENDER_ACCUMULATE, include/rayz_cuda.h): the frame, shard and
// sampling parameters a next batch must repeat, and the samples summed so far.  The device set is the context's own.
struct AccumRecord {
    bool valid = false;
    bool pending = false;   // enqueued by rayz_cuda_render_device(sync = 0): the device error words are not checked yet
    uint32_t width = 0, height = 0, shard_index = 0, shard_count = 1, band_rows = 4, max_depth = 0, moments = 0;
    uint64_t seed = 0;
    float t_min = 0;
    RzCamera cam{};
    uint32_t first_offset = 0;
    uint64_t samples = 0;
};

struct RzContext {
    std::vector<Dev> devs;
    AccumRecord acc;
    bool have_scene = false;
    uint32_t n_spheres = 0;
    RzStats stats{};
    RzStats stage_stats[3]{};   // staged K1: primary kernel / sorted stages / persistent tail kernel (single-kernel variants: all in [0])
    bool stats_valid = false;
    RzTiming timing{};
    RzTuning tun;                 // rayz_cuda_get/set_tuning; defaults in default_tuning()
    uint32_t flags = 0;
    float sb_lo[3] = {0, 0, 0}, sb_hi[3] = {0, 0, 0}, huge_radius = 3.0e38f;   // box of the non-huge spheres (staged K1 sort key / cull)
    // host copy of the sphere boxes: the reference-shaped BVH of K0 is built on first use
    std::vector<double> ref_lo, ref_hi;
    bool ref_built = false;
};

// ------------------------------------------------------------------------------ shard rows
extern "C" uint32_t rayz_cuda_shard_rows(uint32_t height, uint32_t shard_index, uint32_t shard_count, uint32_t band_rows) {
    if (shard_count <= 1) return height;
    if (band_rows == 0) band_rows = 4;
    if (shard_index >= shard_count) return 0;
    const uint32_t n_bands = (height + band_rows - 1) / band_rows;
    uint32_t rows = 0;
    for (uint32_t gb = shard_index; gb < n_bands; gb += shard_count) rows += std::min(band_rows, height - gb * band_rows);
    return rows;
}

extern "C" uint32_t rayz_cuda_context_rows(const RzContext *ctx, uint32_t height, uint32_t shard_index, uint32_t shard_count,
                                           uint32_t band_rows) {
    const uint32_t S = shard_count <= 1 ? 1 : shard_count, s = shard_count <= 1 ? 0 : shard_index;
    const uint32_t nd = ctx ? (uint32_t)ctx->devs.size() : 1u;
    uint32_t rows = 0;
    for (uint32_t d = 0; d < nd; d++) rows += rayz_cuda_shard_rows(height, s * nd + d, S * nd, band_rows ? band_rows : 4);
    return rows;
}

// ------------------------------------------------------------------------------ host-side sphere sets (the tree builders: rz_host_bvh.hpp)
namespace {

struct HostSet {
    std::vector<float4> cr, vel, pkv;
    std::vector<double4> c64, v64;
    std::vector<uint32_t> mat;
    std::vector<int32_t> orig;
    uint32_t n = 0, n_static = 0, n_static_pad = 0, n_pad = 0;
    void push(const RzScene &sc, uint32_t i) {
        const double *c = sc.sphere_center + 3 * i, *v = sc.sphere_velocity + 3 * i;
        const double r = sc.sphere_radius[i];
        cr.push_back(make_float4((float)c[0], (float)c[1], (float)c[2], -(float)(r * r)));
        vel.push_back(make_float4((float)v[0], (float)v[1], (float)v[2], (float)r));
        c64.push_back(make_double4(c[0], c[1], c[2], r));
        v64.push_back(make_double4(v[0], v[1], v[2], 1.0 / r));   // .w = 1 / radius for rz_refine_hit
        mat.push_back(sc.sphere_material[i]);
        orig.push_back((int32_t)i);
    }
    // pair-interleaved copy of cr/vel for the packed FP32x2 search (layout: RzSphereSet::pk)
    std::vector<float4> packed() const {
        std::vector<float4> pk;
        if (n_pad == 0 || (n_static_pad & 1u) || (n_pad & 1u)) return pk;
        for (uint32_t k = 0; k < n_pad; k += 2) {
            const float4 a = cr[k], b = cr[k + 1];
            pk.push_back(make_float4(a.x, b.x, a.y, b.y));
            pk.push_back(make_float4(a.z, b.z, a.w, b.w));
            if (k >= n_static_pad) {
                const float4 va = vel[k], vb = vel[k + 1];
                pk.push_back(make_float4(va.x, vb.x, va.y, vb.y));
                pk.push_back(make_float4(va.z, vb.z, 0.f, 0.f));
            }
        }
        return pk;
    }
    void pad_to(size_t count) {
        while (cr.size() < count) {  // w = -r^2 = +1e30 => nd = |l|^2 + 1e30 > 0 by 20 orders of magnitude more than any rounding: never hit
            cr.push_back(make_float4(0.f, 0.f, 0.f, 1.0e30f));
            vel.push_back(make_float4(0.f, 0.f, 0.f, 0.f));
        }
    }
};

int upload_set(SetBufs &d, const HostSet &h, cudaStream_t s) {
    int rc;
    if ((rc = d.cr.upload(h.cr, s))) return rc;
    if ((rc = d.vel.upload(h.vel, s))) return rc;
    if (!h.pkv.empty() && (rc = d.pk.upload(h.pkv, s))) return rc;
    if ((rc = d.c64.upload(h.c64, s))) return rc;
    if ((rc = d.v64.upload(h.v64, s))) return rc;
    if ((rc = d.mat.upload(h.mat, s))) return rc;
    if ((rc = d.orig.upload(h.orig, s))) return rc;
    d.n = h.n; d.n_static = h.n_static; d.n_static_pad = h.n_static_pad; d.n_pad = h.n_pad;
    return RZ_OK;
}

}  // namespace

// ------------------------------------------------------------------------------ API
static RzTuning default_tuning();
extern "C" uint32_t rayz_cuda_abi_version(void) { return RAYZ_CUDA_ABI_VERSION; }
extern "C" const char *rayz_cuda_last_error(void) { return g_err; }

extern "C" int rayz_cuda_create(const RzConfig *cfg, RzContext **out) {
    if (!out) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return rz_fail(RZ_ERR_CUDA, "rayz_cuda_create: no CUDA device (%s); this backend has no CPU path",
                       e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    int nd = cfg ? cfg->n_devices : 1;
    if (nd <= 0) nd = 1;
    if (nd > 8) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_create: n_devices %d > 8", nd);
    DeviceGuard guard;
    RzContext *ctx = new RzContext();
    ctx->flags = cfg ? cfg->flags : 0u;
    ctx->tun = default_tuning();
    ctx->devs.resize(nd);
    for (int d = 0; d < nd; d++) {
        Dev &D = ctx->devs[d];
        D.id = cfg ? cfg->device_ids[d] : 0;
        if (D.id < 0 || D.id >= count) { delete ctx; return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_create: device id %d out of range (have %d)", D.id, count); }
        for (int q = 0; q < d; q++)
            if (ctx->devs[q].id == D.id) { delete ctx; return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_create: device id %d listed twice", D.id); }
    }
    for (int d = 0; d < nd; d++) {
        Dev &D = ctx->devs[d];
        if ((e = cudaSetDevice(D.id)) != cudaSuccess) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_CUDA, "cudaSetDevice(%d): %s", D.id, cudaGetErrorString(e)); }
        cudaDeviceProp prop;
        if ((e = cudaGetDeviceProperties(&prop, D.id)) != cudaSuccess) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e)); }
        if (prop.major < 10) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library carries sm_100a code only", D.id, prop.major, prop.minor); }
        D.sms = prop.multiProcessorCount;
        if ((e = cudaStreamCreateWithFlags(&D.own_stream, cudaStreamNonBlocking)) != cudaSuccess) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
        D.stream = D.own_stream;
        if ((e = cudaStreamCreateWithFlags(&D.stream2, cudaStreamNonBlocking)) != cudaSuccess || (e = cudaEventCreateWithFlags(&D.ev_s2, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&D.ev_tab, cudaEventDisableTiming)) != cudaSuccess) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
        for (auto &ev : D.ev)
            if ((e = cudaEventCreate(&ev)) != cudaSuccess) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e)); }
        if ((e = rz_path_warm()) != cudaSuccess || (e = rz_bvh_warm()) != cudaSuccess || (e = rz_sort_warm()) != cudaSuccess) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_CUDA, "loading the path kernels: %s", cudaGetErrorString(e)); }
        if (d > 0) {
            // the resolve kernel of device d stores straight into device 0's buffers (NVLink P2P)
            int can = 0;
            cudaDeviceCanAccessPeer(&can, D.id, ctx->devs[0].id);
            if (!can) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_UNSUPPORTED, "device %d cannot access peer %d", D.id, ctx->devs[0].id); }
            e = cudaDeviceEnablePeerAccess(ctx->devs[0].id, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { rayz_cuda_destroy(ctx); return rz_fail(RZ_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e)); }
            cudaGetLastError();
        }
    }
    *out = ctx;
    return RZ_OK;
}

extern "C" void rayz_cuda_destroy(RzContext *ctx) {
    if (!ctx) return;
    DeviceGuard guard;
    for (Dev &D : ctx->devs) {
        if (cudaSetDevice(D.id) != cudaSuccess) continue;
        if (D.own_stream) cudaStreamSynchronize(D.own_stream);
        D.brute.release(); D.bvhset.release(); D.bvh.release(); D.bvh4.release(); D.wide_scratch.release(); D.brute_to_bvh.release(); D.refnodes.release(); D.reforder.release();
        D.c64_orig.release(); D.v64_orig.release(); D.mat_orig.release(); D.lbvh_scratch.release();
        D.m_rec.release(); D.m_kind.release(); D.m_tex.release(); D.m_method.release(); D.t_kind.release(); D.t_even.release(); D.t_odd.release();
        D.m_fuzz.release(); D.m_ior.release(); D.t_color.release(); D.t_inv_scale.release();
        D.accum.release(); D.counter.release(); D.errword.release();
        for (int sd = 0; sd < 2; sd++) { D.q1[sd].release(); D.q2[sd].release(); D.keys[sd].release(); D.idx_sorted[sd].release(); D.bins[sd].release(); }
        D.bin_lists.release();
        D.stats.release(); D.out_linear.release(); D.out_rgb8.release(); D.loc_linear.release(); D.loc_rgb8.release();
        D.out_err.release(); D.noise_part.release();
        D.ids.release(); D.sink.release();
        if (D.wf_scratch) rz_wavefront_free(D.wf_scratch);
        for (auto &ev : D.ev) if (ev) cudaEventDestroy(ev);
        for (auto &ev : D.pass_ev) if (ev) cudaEventDestroy(ev);
        for (auto &ev : D.stage_ev) if (ev) cudaEventDestroy(ev);
        if (D.ev_s2) cudaEventDestroy(D.ev_s2);
        if (D.ev_tab) cudaEventDestroy(D.ev_tab);
        if (D.stream2) { cudaStreamSynchronize(D.stream2); cudaStreamDestroy(D.stream2); }
        if (D.own_stream) cudaStreamDestroy(D.own_stream);
    }
    delete ctx;
}

extern "C" int rayz_cuda_set_stream(RzContext *ctx, void *cuda_stream) {
    if (!ctx) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_set_stream: ctx is NULL");
    Dev &D = ctx->devs[0];
    D.stream = cuda_stream ? (cudaStream_t)cuda_stream : D.own_stream;
    return RZ_OK;
}

// Tuning (include/rayz_cuda.h: RzTuning).  The library reads no environment variables.
static RzTuning default_tuning() {
    RzTuning t;
    memset(&t, 0, sizeof t);
    t.struct_size = (uint32_t)sizeof(RzTuning);
    t.rays_per_thread = 2;
    t.chunk = 16;
    t.chunk_primary = 64;   // the primary kernel builds a culled list per unit: 16 -> 15.9 ms, 32 -> 14.6, 64 -> 14.5, 125 -> 15.3
    t.queue_log2 = 27;
    t.second_stages = -1;
    t.bvh_stages = 0;
    t.tail_brute = 0;
    t.bvh_staged = 1;
    t.cell_bits = 9;
    t.bvh_active_min = 8;
    t.bvh_descend_min = 24;
    t.sah_leaf = 4;
    t.sah_node_cost = 0.5;
    t.unit_entries = 512;
    t.key_sectors = -1;
    t.huge_factor = 4.0;
    t.lbvh_leaf = 1;   // config 4: 1 -> 1872, 2 -> 1848, 3 -> 1844, 4 -> 1735 Mpaths/s (53 box + 1.5 sphere tests per segment against 47 + 6.5)
    return t;
}

extern "C" int rayz_cuda_get_tuning(RzContext *ctx, RzTuning *out) {
    if (!ctx || !out) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_get_tuning: NULL argument");
    *out = ctx->tun;
    return RZ_OK;
}

extern "C" int rayz_cuda_set_tuning(RzContext *ctx, const RzTuning *t) {
    if (!ctx || !t) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_set_tuning: NULL argument");
    if (t->struct_size != sizeof(RzTuning)) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_set_tuning: struct_size %u, expected %zu", t->struct_size, sizeof(RzTuning));
    if (t->rays_per_thread != 1 && t->rays_per_thread != 2) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: rays_per_thread must be 1 or 2");
    if (t->chunk < 1 || t->chunk > 4096 || t->chunk_primary < 1 || t->chunk_primary > 4096) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: chunk out of [1, 4096]");
    if (t->queue_log2 < 16 || t->queue_log2 > 28) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: queue_log2 out of [16, 28]");
    if (t->second_stages < -1 || t->second_stages > 8 || t->bvh_stages < 0 || t->bvh_stages > 8) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: stages out of range");
    if (t->cell_bits < 0 || t->cell_bits > 9) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: cell_bits out of [0, 9]");
    if (t->bvh_active_min < 1 || t->bvh_active_min > 32 || t->bvh_descend_min < 1 || t->bvh_descend_min > 32) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: BVH lane thresholds out of [1, 32]");
    if (t->sah_leaf < 1 || t->sah_leaf > 8 || !(t->sah_node_cost >= 0)) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: SAH parameters out of range");
    if (t->key_sectors < -1 || t->key_sectors > 2) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: key_sectors must be -1, 0, 1 or 2");
    if (t->lbvh_leaf < 1 || t->lbvh_leaf > 8) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: lbvh_leaf out of [1, 8]");
    if (!(t->huge_factor >= 1.0)) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: huge_factor must be >= 1");
    if (t->unit_entries < 64 || t->unit_entries > 2048 || (t->unit_entries & 63u)) return rz_fail(RZ_ERR_INVALID_ARG, "tuning: unit_entries must be a multiple of 64 in [64, 2048]");
    ctx->tun = *t;
    return RZ_OK;
}

static const uint32_t RZ_SMEM_BUDGET = 180u * 1024u;  // of 227 KB per CTA on sm_100: the set, + 25 % for the primary kernel's pair lists

extern "C" int rayz_cuda_upload_scene(RzContext *ctx, const RzScene *sc) {
    if (!ctx || !sc) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_upload_scene: NULL argument");
    ctx->acc.valid = false;   // sums of the old scene: a next batch may not add to them
    const uint32_t n = sc->n_spheres, nm = sc->n_materials, nt = sc->n_textures;
    if (n == 0) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_upload_scene: empty scene (BVH.build asserts nobjs > 0, hit.zig:132)");
    if (n >= (1u << 28)) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_upload_scene: too many spheres (K3 leaf references hold 28 bits)");
    if (!sc->sphere_center || !sc->sphere_velocity || !sc->sphere_radius || !sc->sphere_material || !sc->mat_kind ||
        !sc->mat_fuzz || !sc->mat_ior || !sc->mat_texture || (nt && (!sc->tex_kind || !sc->tex_color || !sc->tex_scale || !sc->tex_even || !sc->tex_odd)))
        return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_upload_scene: NULL array in RzScene");
    for (uint32_t i = 0; i < n; i++) {
        if (sc->sphere_material[i] >= nm) return rz_fail(RZ_ERR_INVALID_ARG, "sphere %u: material %u out of range (%u)", i, sc->sphere_material[i], nm);
        if (!(sc->sphere_radius[i] > 0) || !std::isfinite(sc->sphere_radius[i])) return rz_fail(RZ_ERR_INVALID_ARG, "sphere %u: radius must be finite and > 0", i);
    }
    for (uint32_t i = 0; i < nm; i++) {
        if (sc->mat_kind[i] > 2) return rz_fail(RZ_ERR_INVALID_ARG, "material %u: kind %u", i, sc->mat_kind[i]);
        if (sc->mat_kind[i] != RZ_MAT_DIELECTRIC && sc->mat_texture[i] >= nt) return rz_fail(RZ_ERR_INVALID_ARG, "material %u: texture %u out of range (%u)", i, sc->mat_texture[i], nt);
        if (sc->mat_method && sc->mat_method[i] > 2) return rz_fail(RZ_ERR_INVALID_ARG, "material %u: diffuse method %u", i, sc->mat_method[i]);
    }
    for (uint32_t i = 0; i < nt; i++) {
        if (sc->tex_kind[i] > 1) return rz_fail(RZ_ERR_INVALID_ARG, "texture %u: kind %u", i, sc->tex_kind[i]);
        if (sc->tex_kind[i] == RZ_TEX_CHECKER && (sc->tex_even[i] >= nt || sc->tex_odd[i] >= nt || !(sc->tex_scale[i] != 0)))
            return rz_fail(RZ_ERR_INVALID_ARG, "texture %u: bad checker (even %u, odd %u, scale %g)", i, sc->tex_even[i], sc->tex_odd[i], sc->tex_scale[i]);
    }

    // ---- brute-force set: stationary first (10-instruction test), then moving (13)
    HostSet bs;
    for (uint32_t i = 0; i < n; i++) {
        const double *v = sc->sphere_velocity + 3 * i;
        if (v[0] == 0 && v[1] == 0 && v[2] == 0) bs.push(*sc, i);
    }
    bs.n_static = (uint32_t)bs.cr.size();
    bs.n_static_pad = (bs.n_static + 3u) & ~3u;
    bs.pad_to(bs.n_static_pad);
    // c64/v64/mat/orig are indexed by set position too: keep them aligned with the padding
    auto pad_aux = [](HostSet &h) {
        while (h.c64.size() < h.cr.size()) { h.c64.push_back(make_double4(0, 0, 0, 1)); h.v64.push_back(make_double4(0, 0, 0, 1)); h.mat.push_back(0); h.orig.push_back(-1); }
    };
    pad_aux(bs);
    for (uint32_t i = 0; i < n; i++) {
        const double *v = sc->sphere_velocity + 3 * i;
        if (!(v[0] == 0 && v[1] == 0 && v[2] == 0)) bs.push(*sc, i);
    }
    bs.n = n;
    bs.n_pad = ((uint32_t)bs.cr.size() + 3u) & ~3u;
    bs.pad_to(bs.n_pad);
    pad_aux(bs);
    bs.pkv = bs.packed();

    // ---- spheres in caller order, f64 (K0, LBVH input); boxes kept on the host for the lazy K0 tree
    std::vector<double4> c64o(n), v64o(n);
    std::vector<uint32_t> mato(n);
    ctx->ref_lo.resize(3 * (size_t)n); ctx->ref_hi.resize(3 * (size_t)n);
    ctx->ref_built = false;
    for (uint32_t i = 0; i < n; i++) {
        c64o[i] = make_double4(sc->sphere_center[3 * i], sc->sphere_center[3 * i + 1], sc->sphere_center[3 * i + 2], sc->sphere_radius[i]);
        v64o[i] = make_double4(sc->sphere_velocity[3 * i], sc->sphere_velocity[3 * i + 1], sc->sphere_velocity[3 * i + 2], 0.0);
        mato[i] = sc->sphere_material[i];
        const Box bx = sphere_box(*sc, i);
        for (int a = 0; a < 3; a++) { ctx->ref_lo[3 * (size_t)i + a] = bx.lo[a]; ctx->ref_hi[3 * (size_t)i + a] = bx.hi[a]; }
    }

    // ---- box of the "non-huge" spheres (staged K1): a ray that has left it can only hit a huge sphere (the r = 1000 ground, the three r = 1 spheres: rz_huge_threshold)
    {
        const double huge = rz_huge_threshold(sc->sphere_radius, n, ctx->tun.huge_factor);
        double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
        bool any = false;
        for (uint32_t i = 0; i < n; i++) {
            if (sc->sphere_radius[i] > huge) continue;
            any = true;
            for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], ctx->ref_lo[3 * (size_t)i + a]); hi[a] = std::max(hi[a], ctx->ref_hi[3 * (size_t)i + a]); }
        }
        for (int a = 0; a < 3; a++) {
            const double pad = any ? 1e-3 * (hi[a] - lo[a]) + 1e-3 : 0.0;
            ctx->sb_lo[a] = any ? SahBuilder::down(lo[a] - pad) : -3.0e38f;
            ctx->sb_hi[a] = any ? SahBuilder::up(hi[a] + pad) : 3.0e38f;
        }
        ctx->huge_radius = (float)huge;
    }

    // ---- K3 tree: binned SAH on the host (small scenes) or LBVH on the device (rz_bvh_build.cu)
    const bool device_build = (ctx->flags & RZ_CFG_BVH_BUILD_DEVICE) || (!(ctx->flags & RZ_CFG_BVH_BUILD_HOST) && n >= 8192u);
    SahBuilder sb;
    HostSet vs;
    double host_build_us = 0;
    if (!device_build) {
        const auto t0 = std::chrono::steady_clock::now();
        sb.LEAF = ctx->tun.sah_leaf;
        sb.node_cost = ctx->tun.sah_node_cost;
        sb.p.resize(n);
        for (uint32_t i = 0; i < n; i++) {
            sb.p[i].b = sphere_box(*sc, i);
            for (int a = 0; a < 3; a++) sb.p[i].c[a] = 0.5 * (sb.p[i].b.lo[a] + sb.p[i].b.hi[a]);
            sb.p[i].s = i;
        }
        sb.run();
        for (uint32_t k = 0; k < (uint32_t)sb.order.size(); k++) vs.push(*sc, sb.order[k]);
        vs.n = n; vs.n_static = 0; vs.n_static_pad = 0; vs.n_pad = n;
        host_build_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
    }
    const uint32_t brute_smem = (bs.n_pad * 2 - bs.n_static_pad) * 16u;
    const bool upload_brute = brute_smem <= RZ_SMEM_BUDGET;   // larger scenes can only run the BVH variant
    // staged K1 hands the tail of its paths to the BVH kernel: queue entries name the sphere a ray starts on by its position
    // in the brute-force set, the BVH kernel wants the position in its own (leaf-ordered) set
    std::vector<int32_t> b2v;
    if (!device_build && upload_brute) {
        std::vector<int32_t> pos(n, -1);
        for (uint32_t k = 0; k < (uint32_t)sb.order.size(); k++) pos[sb.order[k]] = (int32_t)k;
        b2v.assign(bs.orig.size(), -1);
        for (size_t j = 0; j < bs.orig.size(); j++) if (bs.orig[j] >= 0) b2v[j] = pos[(size_t)bs.orig[j]];
    }

    // ---- materials / textures
    std::vector<uint32_t> mk(nm), mt(nm), mm(nm), tk(nt), te(nt), to(nt);
    std::vector<float> mf(nm), mi(nm);
    std::vector<float4> tc(nt);
    std::vector<double> ts(nt);
    for (uint32_t i = 0; i < nm; i++) {
        mk[i] = sc->mat_kind[i]; mt[i] = sc->mat_kind[i] == RZ_MAT_DIELECTRIC ? 0u : sc->mat_texture[i];
        mm[i] = sc->mat_method ? sc->mat_method[i] : (uint32_t)RZ_DIFFUSE_HEMISPHERE;
        mf[i] = (float)sc->mat_fuzz[i]; mi[i] = (float)sc->mat_ior[i];
    }
    for (uint32_t i = 0; i < nt; i++) {
        tk[i] = sc->tex_kind[i]; te[i] = sc->tex_even[i]; to[i] = sc->tex_odd[i];
        tc[i] = make_float4((float)sc->tex_color[3 * i], (float)sc->tex_color[3 * i + 1], (float)sc->tex_color[3 * i + 2], 0.f);
        ts[i] = sc->tex_kind[i] == RZ_TEX_CHECKER ? 1.0 / sc->tex_scale[i] : 0.0;
    }
    // the same facts per material in one 64-byte record (RzMaterials::rec)
    std::vector<float4> mrec(4 * (size_t)nm);
    for (uint32_t i = 0; i < nm; i++) {
        const bool textured = mk[i] != RZ_MAT_DIELECTRIC && nt > 0;
        const bool solid = textured && tk[mt[i]] != RZ_TEX_CHECKER;
        const bool checker2 = textured && !solid && tk[te[mt[i]]] != RZ_TEX_CHECKER && tk[to[mt[i]]] != RZ_TEX_CHECKER;
        const uint32_t bits = (mk[i] & 3u) | ((mm[i] & 3u) << 2) | (solid ? 16u : 0u) | (checker2 ? 32u : 0u);
        float fb, ft;
        memcpy(&fb, &bits, 4); memcpy(&ft, &mt[i], 4);
        const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
        mrec[4 * (size_t)i] = make_float4(fb, mf[i], mi[i], ft);
        mrec[4 * (size_t)i + 1] = solid ? tc[mt[i]] : checker2 ? tc[te[mt[i]]] : zero;
        mrec[4 * (size_t)i + 2] = checker2 ? tc[to[mt[i]]] : zero;
        float4 sc4 = zero;
        if (checker2) { const double inv = ts[mt[i]]; uint32_t w[2]; memcpy(w, &inv, 8); memcpy(&sc4.x, &w[0], 4); memcpy(&sc4.y, &w[1], 4); }   // low, high word
        mrec[4 * (size_t)i + 3] = sc4;
    }

    DeviceGuard guard;
    // one host thread per device (as in render_impl): ~25 small copies and allocations each
    auto upload_device = [&](Dev &D) -> int {
        RZ_CUDA(cudaSetDevice(D.id));
        int rc;
        if (upload_brute) { if ((rc = upload_set(D.brute, bs, D.stream))) return rc; }
        else { D.brute.release(); D.brute.n = bs.n; D.brute.n_static = bs.n_static; D.brute.n_static_pad = bs.n_static_pad; D.brute.n_pad = bs.n_pad; }
        if ((rc = D.c64_orig.upload(c64o, D.stream))) return rc;
        if ((rc = D.v64_orig.upload(v64o, D.stream))) return rc;
        if ((rc = D.mat_orig.upload(mato, D.stream))) return rc;
        if (b2v.empty()) D.brute_to_bvh.release();
        if (!device_build) {
            if ((rc = upload_set(D.bvhset, vs, D.stream))) return rc;
            if ((rc = D.bvh.upload(sb.nodes, D.stream))) return rc;
            D.bvh_nodes = (uint32_t)sb.nodes.size();
            if (!b2v.empty() && (rc = D.brute_to_bvh.upload(b2v, D.stream))) return rc;
        } else {
            const size_t scratch = rz_lbvh_scratch_bytes(n);
            if ((rc = D.lbvh_scratch.alloc(scratch))) return rc;
            SetBufs &V = D.bvhset;
            if ((rc = V.cr.alloc(n)) || (rc = V.vel.alloc(n)) || (rc = V.c64.alloc(n)) || (rc = V.v64.alloc(n)) || (rc = V.mat.alloc(n)) ||
                (rc = V.orig.alloc(n)))
                return rc;
            V.n = n; V.n_static = 0; V.n_static_pad = 0; V.n_pad = n;
            D.bvh_nodes = n > 1 ? n - 1 : 1;
            if ((rc = D.bvh.alloc(D.bvh_nodes))) return rc;
            RZ_CUDA(cudaEventRecord(D.ev[0], D.stream));
            RZ_CUDA(rz_lbvh_build(n, ctx->tun.lbvh_leaf, D.c64_orig.p, D.v64_orig.p, D.mat_orig.p, D.lbvh_scratch.p, D.lbvh_scratch.n, D.bvh.p, V.cr.p, V.vel.p,
                                  V.c64.p, V.v64.p, V.mat.p, V.orig.p, D.stream));
        }
#ifdef RZ_BVH_WIDE   // experiment: K3 walks the 4-wide collapse of the builders' binary tree (three small kernels, no host round trip)
        if ((rc = D.bvh4.alloc(D.bvh_nodes)) || (rc = D.wide_scratch.alloc(rz_bvh_wide_scratch_bytes(D.bvh_nodes) / sizeof(int)))) return rc;
        RZ_CUDA(rz_bvh_wide_collapse(D.bvh.p, D.bvh_nodes, D.wide_scratch.p, D.bvh4.p, D.stream));
#else
        RZ_CUDA(rz_bvh_finalize(D.bvh.p, D.bvh_nodes, D.stream));   // leaves -> the references K3 follows; no unused slots
#endif
        if (device_build) RZ_CUDA(cudaEventRecord(D.ev[1], D.stream));
        if ((rc = D.m_rec.upload(mrec, D.stream)) || (rc = D.m_kind.upload(mk, D.stream)) || (rc = D.m_tex.upload(mt, D.stream)) || (rc = D.m_method.upload(mm, D.stream)) ||
            (rc = D.m_fuzz.upload(mf, D.stream)) || (rc = D.m_ior.upload(mi, D.stream)) || (rc = D.t_kind.upload(tk, D.stream)) ||
            (rc = D.t_even.upload(te, D.stream)) || (rc = D.t_odd.upload(to, D.stream)) || (rc = D.t_color.upload(tc, D.stream)) ||
            (rc = D.t_inv_scale.upload(ts, D.stream)))
            return rc;
        return RZ_OK;
    };
    if (ctx->devs.size() == 1) {
        const int rc = upload_device(ctx->devs[0]);
        if (rc) return rc;
    } else {
        const size_t nd = ctx->devs.size();
        std::vector<int> rcs(nd, RZ_OK);
        std::vector<std::string> errs(nd);
        std::vector<std::thread> workers;
        workers.reserve(nd);
        for (size_t d = 0; d < nd; d++)
            workers.emplace_back([&, d] { rcs[d] = upload_device(ctx->devs[d]); if (rcs[d]) errs[d] = g_err; });
        for (std::thread &w : workers) w.join();
        for (size_t d = 0; d < nd; d++)
            if (rcs[d]) return rz_fail(rcs[d], "%s", errs[d].c_str());
    }
    for (Dev &D : ctx->devs) {   // every device's copies are in flight before the first wait
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaStreamSynchronize(D.stream));  // host vectors die at return: copy semantics
        if (device_build) {
            float ms = 0;
            RZ_CUDA(cudaEventElapsedTime(&ms, D.ev[0], D.ev[1]));
            host_build_us = std::max(host_build_us, (double)ms * 1e3);
        }
    }
    ctx->timing.bvh_build_us = (uint32_t)std::min(host_build_us, 4.0e9);
    ctx->have_scene = true;
    ctx->n_spheres = n;
    ctx->timing.n_static = bs.n_static;
    ctx->timing.n_moving = n - bs.n_static;
    return RZ_OK;
}

static RzCamF32 cam_to_f32(const RzCamera *c) {
    RzCamF32 k;
    k.look_from = make_float3((float)c->look_from[0], (float)c->look_from[1], (float)c->look_from[2]);
    k.px_du = make_float3((float)c->px_du[0], (float)c->px_du[1], (float)c->px_du[2]);
    k.px_dv = make_float3((float)c->px_dv[0], (float)c->px_dv[1], (float)c->px_dv[2]);
    k.px_origin = make_float3((float)c->px_origin[0], (float)c->px_origin[1], (float)c->px_origin[2]);
    k.defocus_u = make_float3((float)c->defocus_u[0], (float)c->defocus_u[1], (float)c->defocus_u[2]);
    k.defocus_v = make_float3((float)c->defocus_v[0], (float)c->defocus_v[1], (float)c->defocus_v[2]);
    k.defocus = c->defocus;
    return k;
}


// Pass/queue sizing of the staged K1 (see render_impl).
struct QueuePlan {
    uint64_t unit_paths = 0, cap = 0;
    uint32_t units_per_pass = 1, n_pass = 1;
    int n_sides = 1, n_second = 0;
    bool second_stage = false;
};

static QueuePlan plan_queues(const RzTuning &tun, uint32_t n_units, uint32_t chunk, bool serial, bool enough_spheres, bool bvh_family, bool bvh_tail,
                             int qlog_cap) {
    QueuePlan q;
    q.unit_paths = 32ull * chunk;
    // Queue size = pass size.  Measured at config 2 (405 M paths, round 1): 2^26 -> 5140, 2^27 -> 5405, 2^28 -> 5529 Mpaths/s
    // (fewer, longer launches; fewer tails).  The default is 2^27 entries (RzTuning::queue_log2): 6.4 GB per queue buffer,
    // ~31 GB for both sides with keys and indices; plan_and_alloc_queues steps down if the device cannot give that much.
    const int qlog = std::min(qlog_cap, tun.queue_log2);
    // Sorted stages after the camera segment, measured in round 1 (Mpaths/s, config 2 / glass-heavy scene), BVH tail:
    // 3 -> 5426 / 4025, 4 -> 5510 / 4130, 5 -> 5549 / 4214, 6 -> 5547 / 4264; brute-force tail: 3 -> 3634 / 2635, 4 -> 3648 /
    // 2797, 5 -> 3576 / 2899.  BVH family: sorted stages measured as a loss (config-2 scene 3521 -> 3277 -> 3065 Mpaths/s for
    // 0, 1, 2 stages; 100k spheres 1582 -> 1427 -> 1327): batches without in-loop ray replacement cost more than coherence
    // gains; only the coherent camera stage is kept.  Round 2, after the sorted-stage kernel got ~25 % cheaper per segment
    // (profiles/r02_experiments.md, exp23; BVH tail): 4 -> 6439 / 4648, 5 -> 6575 / 4806, 6 -> 6667 / 4920, 7 -> 6713 / 4941.
    // NOTE: none of this depends on the job's size, shard count or on how much memory the device had left, so that a sharded
    // render runs exactly the kernels — and therefore computes exactly the pixels — of the full-frame one.
    if (bvh_family) q.n_second = enough_spheres ? tun.bvh_stages : 0;
    else q.n_second = !enough_spheres ? 0 : tun.second_stages >= 0 ? tun.second_stages : !bvh_tail ? 4 : 7;
    q.cap = std::max<uint64_t>(q.unit_paths, std::min<uint64_t>((uint64_t)n_units * q.unit_paths, 1ull << qlog));
    q.second_stage = q.n_second > 0;
    q.units_per_pass = (uint32_t)std::max<uint64_t>(1, q.cap / q.unit_paths);
    q.n_pass = (n_units + q.units_per_pass - 1) / q.units_per_pass;
    // Passes alternate between two streams so that the next pass's first kernel fills the tail of the persistent one — except for
    // K3 with tile lists: its camera stage holds 41 KB of shared memory per CTA, and running beside the traversal kernel of the
    // previous pass it takes the L1 that kernel's node loads live in (config 4: 247.6 ms overlapped against 212.6 ms in series).
    const bool overlap = !(bvh_family && rz_bvh_camera_tile_w() != 0u);
    q.n_sides = (q.n_pass > 1 && !serial && overlap) ? 2 : 1;
    return q;
}

static int alloc_queues(Dev &D, const QueuePlan &q) {
    int rc;
    for (int sd = 0; sd < q.n_sides; sd++) {
        if ((rc = D.q1[sd].alloc((size_t)q.cap * 4u))) return rc;
        if (q.second_stage) {
            if ((rc = D.q2[sd].alloc((size_t)q.cap * 4u)) || (rc = D.keys[sd].alloc((size_t)q.cap)) ||
                (rc = D.idx_sorted[sd].alloc((size_t)q.cap)) || (rc = D.bins[sd].alloc(rz_bin_scratch_bytes() / sizeof(unsigned int))))
                return rc;
        }
    }
    return RZ_OK;
}

// Plans the passes and allocates their queues; when the device cannot give the memory (others share it, or a smaller part),
// the plan is redone with queues half the size, down to 2^22 entries.  Only the pass size changes, never which kernels run.
static int plan_and_alloc_queues(const RzTuning &tun, Dev &D, QueuePlan &qp, uint32_t n_units, uint32_t chunk, bool serial, bool enough_spheres,
                                 bool bvh_family, bool bvh_tail) {
    for (int qlog = 28;; qlog--) {
        qp = plan_queues(tun, n_units, chunk, serial, enough_spheres, bvh_family, bvh_tail, qlog);
        const int rc = alloc_queues(D, qp);
        if (rc != RZ_ERR_OOM || qlog <= 22 || qp.cap < (1ull << qlog)) return rc;   // done, a real error, or nothing left to shrink
        cudaGetLastError();
        for (int sd = 0; sd < 2; sd++) {
            D.q1[sd].release(); D.q2[sd].release(); D.keys[sd].release(); D.idx_sorted[sd].release();
        }
    }
}

// Device timings (CUDA events) and, if asked for, the counters of the render that just finished on every stream.
static int collect_timing_and_stats(RzContext *ctx, bool collect_stats) {
    float kmax = 0, rmax = 0, pmax = 0, smax = 0, somax = 0;
    uint32_t passes = 0;
    for (Dev &D : ctx->devs) {
        float k = 0, r = 0, pr = 0, se = 0, so = 0;
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaEventElapsedTime(&k, D.ev[1], D.ev[2]));
        RZ_CUDA(cudaEventElapsedTime(&r, D.ev[2], D.ev[3]));
        for (uint32_t i = 0; i < D.passes; i++) {
            // overlapped: pass i runs on stream i & 1 after pass i-2 of that stream (the first two start at ev[1]); serial: after pass i-1
            const uint32_t back = D.serial_passes ? 1u : 2u;
            float ms = 0;
            RZ_CUDA(cudaEventElapsedTime(&ms, i < back ? D.ev[1] : D.pass_ev[3 * (i - back) + 2], D.pass_ev[3 * i]));
            pr += ms;
            for (uint32_t g = 0; g < D.n_second; g++) {   // sort, then the sorted-segment kernel
                const size_t b = 2 * ((size_t)i * D.n_second + g);
                RZ_CUDA(cudaEventElapsedTime(&ms, g == 0 ? D.pass_ev[3 * i] : D.stage_ev[b - 1], D.stage_ev[b]));
                so += ms;
                RZ_CUDA(cudaEventElapsedTime(&ms, D.stage_ev[b], D.stage_ev[b + 1]));
                se += ms;
            }
        }
        kmax = std::max(kmax, k); rmax = std::max(rmax, r); pmax = std::max(pmax, pr); smax = std::max(smax, se); somax = std::max(somax, so);
        passes = std::max(passes, D.passes);
    }
    for (Dev &D : ctx->devs) {   // a device-side capacity was exceeded: work was dropped, the result is not to be used
        unsigned int ew = 0;
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaMemcpy(&ew, D.errword.p, sizeof ew, cudaMemcpyDeviceToHost));
        if (ew) return rz_fail(RZ_ERR_INTERNAL, "render: device %d reported%s%s (error word 0x%x): paths were dropped, result withheld", D.id,
                               (ew & RZ_DEV_ERR_QUEUE_OVERFLOW) ? " a queue overflow" : "", (ew & RZ_DEV_ERR_STACK_OVERFLOW) ? " a traversal-stack overflow" : "", ew);
    }
    ctx->timing.kernel_ms = kmax;
    ctx->timing.resolve_ms = rmax;
    ctx->timing.primary_ms = pmax;
    ctx->timing.second_ms = smax;
    ctx->timing.sort_ms = somax;
    ctx->timing.passes = passes;
    ctx->timing.sorted_stages = ctx->devs[0].n_second;
    ctx->timing.queue_entries = ctx->devs[0].queue_entries;
    if (collect_stats) {
        RzStats tot, stage[3];
        memset(&tot, 0, sizeof tot);
        memset(stage, 0, sizeof stage);
        for (Dev &D : ctx->devs) {
            RzStatsDev h[3];
            RZ_CUDA(cudaSetDevice(D.id));
            RZ_CUDA(cudaMemcpy(h, D.stats.p, sizeof h, cudaMemcpyDeviceToHost));
            for (int k = 0; k < 3; k++) {
                RzStats *dst[2] = {&tot, &stage[k]};
                for (RzStats *t : dst) {
                    t->paths += h[k].v[0]; t->segments += h[k].v[1]; t->sphere_tests += h[k].v[2]; t->node_tests += h[k].v[3];
                    t->hits_diffuse += h[k].v[4]; t->hits_metallic += h[k].v[5]; t->hits_dielectric += h[k].v[6];
                    t->ended_sky += h[k].v[7]; t->ended_absorbed += h[k].v[8]; t->ended_depth += h[k].v[9];
                }
            }
        }
        ctx->stats = tot;
        for (int k = 0; k < 3; k++) ctx->stage_stats[k] = stage[k];
        ctx->stats_valid = true;
    }
    return RZ_OK;
}

// An accumulation left pending by rayz_cuda_render_device(sync = 0): wait for it and read the device error words, so that a
// batch that dropped paths ends the accumulation before anything is added to its sums.
static int settle_accumulation(RzContext *ctx) {
    if (!ctx->acc.valid || !ctx->acc.pending) return RZ_OK;
    ctx->acc.valid = false;
    for (Dev &D : ctx->devs) {
        unsigned int ew = 0;
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaStreamSynchronize(D.stream));
        RZ_CUDA(cudaMemcpy(&ew, D.errword.p, sizeof ew, cudaMemcpyDeviceToHost));
        if (ew) return RZ_OK;   // stays invalid
    }
    ctx->acc.valid = true;
    ctx->acc.pending = false;
    return RZ_OK;
}

static int render_impl(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, bool sync, bool host_direct = false) {
    if (!ctx || !cam || !p) return rz_fail(RZ_ERR_INVALID_ARG, "render: NULL argument");
    // Every render ends what the accumulators held unless it succeeds (the record is committed at the end) or it is an
    // RZ_RENDER_ACCUMULATE batch that is refused before anything was touched (the record is restored).
    const bool accumulate = (p->flags & RZ_RENDER_ACCUMULATE) != 0;
    if (accumulate) { DeviceGuard g; const int rc = settle_accumulation(ctx); if (rc) return rc; }
    const AccumRecord prev = ctx->acc;
    ctx->acc.valid = false;
    if (!ctx->have_scene) return rz_fail(RZ_ERR_NO_SCENE, "render: rayz_cuda_upload_scene has not been called");
    if (p->width == 0 || p->height == 0 || p->spp == 0) return rz_fail(RZ_ERR_INVALID_ARG, "render: width, height and spp must be > 0");
    if ((uint64_t)p->width * p->height >= (1ull << 31)) return rz_fail(RZ_ERR_INVALID_ARG, "render: image too large");
    const uint32_t S = p->shard_count <= 1 ? 1 : p->shard_count;
    const uint32_t s = p->shard_count <= 1 ? 0 : p->shard_index;
    if (s >= S) return rz_fail(RZ_ERR_INVALID_ARG, "render: shard_index %u >= shard_count %u", s, S);
    const uint32_t band = p->band_rows ? p->band_rows : 4;
    const uint32_t ND = (uint32_t)ctx->devs.size();
    uint32_t variant = p->variant;
    const uint32_t brute_smem = (ctx->devs[0].brute.n_pad * 2 - ctx->devs[0].brute.n_static_pad) * 16u;
    if (variant == RZ_VARIANT_AUTO) {
        // AUTO picks by cost: the staged brute-force K1 when the sphere set fits shared memory AND the frame is big enough to
        // amortise its ~25 launches per pass (measured one-shot, 485 spheres: 0.9 M paths 3.9 ms vs 0.8 ms for the BVH kernel,
        // 8 M 6.3 vs 2.8, 81 M 23.8 vs 25.3, 405 M 104 vs 125); else the BVH kernel.  The choice looks at the WHOLE FRAME
        // (width x height x spp), never at this shard's or device's share of it: every shard of a frame runs the same
        // kernels, so a sharded render equals the full-frame one bit for bit (the two kernel families themselves can
        // differ in a pixel or two: FP32 sphere test against exact boxes, tests/test_gpu_parity.py).
        const uint64_t frame_paths = (uint64_t)p->width * p->height * p->spp;
        variant = (brute_smem <= RZ_SMEM_BUDGET && frame_paths >= (1ull << 26)) ? RZ_VARIANT_MEGA : RZ_VARIANT_BVH;
    }
    const bool mega_single = variant == RZ_VARIANT_MEGA_SINGLE;
    if (mega_single) variant = RZ_VARIANT_MEGA;
    if (variant != RZ_VARIANT_MEGA && variant != RZ_VARIANT_BVH && variant != RZ_VARIANT_WAVEFRONT)
        return rz_fail(RZ_ERR_INVALID_ARG, "render: unknown variant %u", p->variant);
    if (variant == RZ_VARIANT_MEGA && brute_smem > RZ_SMEM_BUDGET)
        return rz_fail(RZ_ERR_UNSUPPORTED, "render: scene needs %u B of shared memory for the brute-force kernel (budget %u); use RZ_VARIANT_BVH", brute_smem, RZ_SMEM_BUDGET);

    AccumRecord next;
    next.width = p->width; next.height = p->height; next.shard_index = s; next.shard_count = S; next.band_rows = band;
    next.max_depth = p->max_depth; next.moments = (p->flags & RZ_RENDER_MOMENTS) ? 1u : 0u; next.seed = p->seed;
    next.t_min = p->t_min > 0 ? p->t_min : 1e-4f; next.cam = *cam;
    next.first_offset = p->sample_offset; next.samples = p->spp;
    if (accumulate) {
        auto refuse = [&](const char *why) { ctx->acc = prev; return rz_fail(RZ_ERR_INVALID_ARG, "render: RZ_RENDER_ACCUMULATE refused: %s", why); };
        if (!prev.valid) return refuse("no previous render to add to (none, it failed, or a scene upload or reserve came in between)");
        if (prev.width != next.width || prev.height != next.height || prev.shard_index != s || prev.shard_count != S || prev.band_rows != band)
            return refuse("frame size, shard or band_rows differ from the accumulated render");
        if (prev.seed != next.seed || prev.max_depth != next.max_depth || memcmp(&prev.t_min, &next.t_min, sizeof(float)) != 0)
            return refuse("seed, max_depth or t_min differ from the accumulated render");
        if (memcmp(&prev.cam, cam, sizeof(RzCamera)) != 0) return refuse("the camera differs from the accumulated render");
        if (prev.moments != next.moments) return refuse("the RZ_RENDER_MOMENTS bit differs from the accumulated render");
        if ((uint64_t)p->sample_offset != (uint64_t)prev.first_offset + prev.samples)
            return refuse("sample_offset must continue where the accumulated samples end (previous sample_offset + spp)");
        if (prev.samples + p->spp > 0xFFFFFFFFull) return refuse("the cumulative sample count would pass 2^32 - 1");
        next.first_offset = prev.first_offset;
        next.samples = prev.samples + p->spp;
    }

    const auto t_host0 = std::chrono::steady_clock::now();
    DeviceGuard guard;
    const uint32_t rows_ctx = [&] { uint32_t r = 0; for (uint32_t d = 0; d < ND; d++) r += rayz_cuda_shard_rows(p->height, s * ND + d, S * ND, band); return r; }();
    Dev &D0 = ctx->devs[0];
    RZ_CUDA(cudaSetDevice(D0.id));
    if (!host_direct) {
        int rc;
        if ((rc = D0.out_linear.alloc((size_t)rows_ctx * p->width))) return rc;
        if ((rc = D0.out_rgb8.alloc((size_t)rows_ctx * p->width * 3))) return rc;
    }
    // Everything one device needs for this render, enqueued on its streams.  A context with several devices runs this on one
    // host thread PER DEVICE: ~90 launches per pass and device issued from a single thread made device 7 start milliseconds
    // after device 0 (e2e 5 % below the device-resident rate at 8 GPUs).
    std::vector<uint32_t> launches_dev(ND, 0u);
    auto per_device = [&](uint32_t d) -> int {
        uint32_t &launches = launches_dev[d];
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        const uint32_t sh_index = s * ND + d, sh_count = S * ND;
        const uint32_t rows = rayz_cuda_shard_rows(p->height, sh_index, sh_count, band);
        const uint32_t n_local = rows * p->width;
        const uint32_t n_tiles = (n_local + 31u) / 32u;
        int rc;
        if ((rc = D.accum.alloc((size_t)n_tiles * 32u * 4u))) return rc;
        if ((rc = D.counter.alloc(16)) || (rc = D.errword.alloc(4))) return rc;
        if ((rc = D.stats.alloc(3))) return rc;   // [0] whole render / primary kernel, [1] sorted stages, [2] persistent tail kernel
        RZ_CUDA(cudaEventRecord(D.ev[0], D.stream));
        if (!accumulate) RZ_CUDA(cudaMemsetAsync(D.accum.p, 0, (size_t)n_tiles * 32u * 4u * sizeof(unsigned long long), D.stream));
        RZ_CUDA(cudaMemsetAsync(D.counter.p, 0, 16 * sizeof(unsigned int), D.stream));
        RZ_CUDA(cudaMemsetAsync(D.errword.p, 0, 4 * sizeof(unsigned int), D.stream));
        if (p->collect_stats) RZ_CUDA(cudaMemsetAsync(D.stats.p, 0, 3 * sizeof(RzStatsDev), D.stream));

        RzPathArgs a;
        memset(&a, 0, sizeof a);
        a.set = (variant == RZ_VARIANT_BVH) ? D.bvhset.view() : D.brute.view();
        a.mats.kind = D.m_kind.p; a.mats.fuzz = D.m_fuzz.p; a.mats.ior = D.m_ior.p; a.mats.tex = D.m_tex.p; a.mats.method = D.m_method.p; a.mats.rec = D.m_rec.p;
        a.texs.kind = D.t_kind.p; a.texs.color = D.t_color.p; a.texs.inv_scale = D.t_inv_scale.p; a.texs.even = D.t_even.p; a.texs.odd = D.t_odd.p;
#ifdef RZ_BVH_WIDE
        a.bvh = D.bvh4.p; a.bvh_nodes = D.bvh_nodes;
#else
        a.bvh = D.bvh.p; a.bvh_nodes = D.bvh_nodes;
#endif
        a.cam = cam_to_f32(cam);
        a.accum = D.accum.p; a.unit_counter = D.counter.p; a.stats = D.stats.p;
        a.width = p->width; a.height = p->height; a.n_local_px = n_local;
        a.spp = p->spp; a.sample_offset = p->sample_offset; a.max_depth = p->max_depth;
        a.chunk = std::min(ctx->tun.chunk, p->spp);
        a.n_chunks = (p->spp + a.chunk - 1) / a.chunk;
        if ((uint64_t)n_tiles * a.n_chunks >= (1ull << 32)) return rz_fail(RZ_ERR_INVALID_ARG, "render: too many work units");
        a.n_units = n_tiles * a.n_chunks;
        a.shard_index = sh_index; a.shard_count = sh_count; a.band_rows = band;
        a.seed_lo = (uint32_t)p->seed; a.seed_hi = (uint32_t)(p->seed >> 32);
        a.t_min = p->t_min > 0 ? p->t_min : 1e-4f;
        a.err = D.errword.p;
        a.unit_entries = ctx->tun.unit_entries;
        a.bvh_active_min = (uint32_t)ctx->tun.bvh_active_min; a.bvh_descend_min = (uint32_t)ctx->tun.bvh_descend_min;
        a.stack_cap = ctx->tun.debug_stack_cap;   // 0 = the kernel's own RZ_STACK
        a.moments = next.moments;

        RZ_CUDA(cudaEventRecord(D.ev[1], D.stream));
        D.passes = 0;
        D.n_second = 0;
        D.queue_entries = 0;
        if (n_local > 0) {
            if (variant == RZ_VARIANT_WAVEFRONT) {
                uint32_t l = 0;
                RZ_CUDA(rz_wavefront_render(&a, D.sms, (int)p->collect_stats, D.stream, &D.wf_scratch, &D.wf_scratch_bytes, &l));
                launches += l;
            } else {
                // K3 on a big job: the same staged pipeline with BVH traversal instead of culled lists (sorted rays stay converged)
                const bool bvh_family = variant == RZ_VARIANT_BVH;
                const bool bvh_staged = bvh_family && ctx->tun.bvh_staged && (uint64_t)p->width * p->height * p->spp >= (1ull << 26);   // by the FRAME's size, never a shard's: every shard of a frame runs the same kernels (the staged camera stage searches block lists, the unstaged kernel walks the tree)
                if (bvh_family && !bvh_staged) {
                    RZ_CUDA(rz_launch_bvh(&a, (int)p->collect_stats, D.sms, D.stream));
                    launches += 1;
                } else if (!bvh_family && (mega_single || rz_primary_smem_bytes(&a) > 227u * 1024u)) {
                    // one persistent kernel (RZ_VARIANT_MEGA_SINGLE, or a set whose pair lists do not fit beside it)
                    RZ_CUDA(rz_launch_path(&a, ctx->tun.rays_per_thread, (int)p->collect_stats, D.sms, D.stream, nullptr));
                    launches += 1;
                } else {
                    // staged K1: primary kernel (tile-culled camera segments) -> queue -> [sort -> sorted-segment kernel (culled per
                    // unit) -> queue] x n_second -> persistent tail kernel (BVH, or brute force).  Passes are sized by the queues
                    // (RzTuning::queue_log2, default 2^27 entries per buffer; two buffers per side, two sides).
                    const bool serial = (p->flags & RZ_RENDER_SERIAL_PASSES) != 0;
                    {   // the camera-stage kernels build a culled sphere list per unit: their own, larger work-unit size
                        a.chunk = std::min(ctx->tun.chunk_primary, p->spp);
                        a.n_chunks = (p->spp + a.chunk - 1) / a.chunk;
                        uint64_t tiles = n_tiles;
                        if (bvh_family && rz_bvh_camera_tile_w()) {   // K3's camera stage works on 8 x 4 pixel blocks
                            a.tile_w = rz_bvh_camera_tile_w();
                            tiles = (uint64_t)((p->width + 7u) / 8u) * ((n_local / p->width + 3u) / 4u);
                        }
                        if (tiles * a.n_chunks >= (1ull << 32)) return rz_fail(RZ_ERR_INVALID_ARG, "render: too many work units");
                        a.n_units = (uint32_t)tiles * a.n_chunks;
                    }
                    // The tail of the paths (whatever survives the sorted stages: incoherent, few) goes to the BVH kernel when the
                    // host-built tree is there — ~28 node + sphere tests per segment instead of every sphere of the set
                    // (config 2: 29.2 -> 11.1 ms behind four sorted stages).
                    const bool bvh_tail = !bvh_family && D.brute_to_bvh.p != nullptr && !ctx->tun.tail_brute;
                    QueuePlan qp;
                    if ((rc = plan_and_alloc_queues(ctx->tun, D, qp, a.n_units, a.chunk, serial, ctx->n_spheres >= 64u, bvh_family, bvh_tail))) return rc;
                    const uint64_t unit_paths = qp.unit_paths, cap = qp.cap;
                    const uint32_t units_per_pass = qp.units_per_pass, total_units = a.n_units, n_pass = qp.n_pass;
                    const int n_sides = qp.n_sides, n_second = qp.n_second;
                    const bool second_stage = qp.second_stage;
                    const double pcx = cam->px_origin[0] + 0.5 * (p->width - 1) * cam->px_du[0] + 0.5 * (p->height - 1) * cam->px_dv[0] - cam->look_from[0];
                    const double pcy = cam->px_origin[1] + 0.5 * (p->width - 1) * cam->px_du[1] + 0.5 * (p->height - 1) * cam->px_dv[1] - cam->look_from[1];
                    const double pcz = cam->px_origin[2] + 0.5 * (p->width - 1) * cam->px_du[2] + 0.5 * (p->height - 1) * cam->px_dv[2] - cam->look_from[2];
                    a.focus_dist = (float)std::sqrt(pcx * pcx + pcy * pcy + pcz * pcz);   // look_from -> centre of the focus plane
                    const double lu = std::sqrt(cam->defocus_u[0] * cam->defocus_u[0] + cam->defocus_u[1] * cam->defocus_u[1] + cam->defocus_u[2] * cam->defocus_u[2]);
                    const double lv = std::sqrt(cam->defocus_v[0] * cam->defocus_v[0] + cam->defocus_v[1] * cam->defocus_v[1] + cam->defocus_v[2] * cam->defocus_v[2]);
                    a.lens_radius = cam->defocus ? (float)(std::max(lu, lv) * 1.001) : 0.f;
                    a.queue_cap = ctx->tun.debug_queue_cap ? std::min((uint32_t)cap, ctx->tun.debug_queue_cap) : (uint32_t)cap;
                    rz_key_grid(a, ctx->sb_lo, ctx->sb_hi, ctx->tun.cell_bits, ctx->tun.key_sectors);
                    a.huge_radius = ctx->huge_radius;
                    uint32_t ue_div = 0;
                    if (second_stage && !bvh_family) {
                        // the sorted-segment kernel's pair lists, one row per sort group: a function of the set and the key grid
                        a.bin_row = rz_bin_row_bytes(a.set.n_pad);
                        if (int rc = D.bin_lists.alloc((size_t)RZ_SORT_BINS * a.bin_row)) return rc;
                        a.bin_lists = D.bin_lists.p;
                        RZ_CUDA(rz_launch_bin_lists(&a, D.sms, D.stream));
                        launches += 1;
                        int grid2 = 0;
                        RZ_CUDA(rz_second_grid(&a, (int)p->collect_stats, D.sms, &grid2));
                        ue_div = 16u * (uint32_t)grid2;
                    }
                    RZ_CUDA(cudaEventRecord(D.ev_tab, D.stream));
                    while (D.pass_ev.size() < 3 * (size_t)n_pass) {
                        cudaEvent_t e = nullptr;
                        RZ_CUDA(cudaEventCreate(&e));
                        D.pass_ev.push_back(e);
                    }
                    while (D.stage_ev.size() < 2 * (size_t)n_pass * (size_t)n_second) {
                        cudaEvent_t e = nullptr;
                        RZ_CUDA(cudaEventCreate(&e));
                        D.stage_ev.push_back(e);
                    }
                    D.passes = n_pass;
                    D.n_second = (uint32_t)n_second;
                    D.queue_entries = (uint32_t)cap;
                    D.serial_passes = serial;
                    // Passes alternate between two streams and two sets of buffers: the persistent kernel ends with a tail of a
                    // few long paths (measured ~2 ms per pass), which the next pass's kernels fill.
                    if (n_sides > 1) RZ_CUDA(cudaStreamWaitEvent(D.stream2, D.ev_tab, 0));   // (recorded after ev[1] on the same stream)
                    uint32_t pass = 0;
                    for (uint32_t u0 = 0; u0 < total_units; u0 += units_per_pass, pass++) {
                        const int side = n_sides > 1 ? (int)(pass & 1u) : 0;
                        cudaStream_t st = side ? D.stream2 : D.stream;
                        unsigned int *ctr = D.counter.p + 8 * side;   // [0..2] unit counters of K1a/K1c/K1b, [3] entries in q1, [4] entries in q2
                        if (pass >= (uint32_t)n_sides) RZ_CUDA(cudaMemsetAsync(ctr, 0, 8 * sizeof(unsigned int), st));
                        const uint32_t pass_units = std::min(units_per_pass, total_units - u0);
                        RzPathArgs a1 = a;
                        a1.q_out = D.q1[side].p; a1.q_out_count = ctr + 3; a1.q_out_keys = second_stage ? D.keys[side].p : nullptr;
                        a1.unit_base = u0; a1.n_units = pass_units; a1.unit_counter = ctr;
                        if (bvh_family) RZ_CUDA(rz_launch_bvh_stage(&a1, (int)p->collect_stats, D.sms, st));
                        else RZ_CUDA(rz_launch_primary(&a1, (int)p->collect_stats, D.sms, st));
                        RZ_CUDA(cudaEventRecord(D.pass_ev[3 * pass], st));
                        launches += 1;
                        RzPathArgs a3 = a;
                        a3.q_in = D.q1[side].p; a3.q_in_count = ctr + 3;
                        // sorted, culled stages for the next `n_second` segments: q1 -> q2 -> q1 -> ...
                        float4 *qa = D.q1[side].p, *qb = second_stage ? D.q2[side].p : nullptr;
                        unsigned int *ca = ctr + 3, *cb = ctr + 4;
                        for (int stg = 0; stg < n_second; stg++) {
                            const bool more = stg + 1 < n_second;
                            // group the entries by key (rz_sort.cu: count / scan / scatter, sized on the device from the live count)
                            RZ_CUDA(rz_bin_sort(D.keys[side].p, ca, a.queue_cap, D.bins[side].p, nullptr, D.idx_sorted[side].p, a.unit_entries, ue_div, D.sms, st));
                            RZ_CUDA(cudaEventRecord(D.stage_ev[2 * ((size_t)pass * n_second + stg)], st));
                            if (stg > 0) RZ_CUDA(cudaMemsetAsync(cb, 0, sizeof(unsigned int), st));           // recycled output counter
                            if (stg > 0) RZ_CUDA(cudaMemsetAsync(ctr + 1, 0, sizeof(unsigned int), st));      // the stage's unit counter
                            RzPathArgs a2 = a;
                            a2.q_in = qa; a2.q_in_count = ca; a2.q_in_idx = D.idx_sorted[side].p; a2.q_in_bins = D.bins[side].p;
                            a2.q_out = qb; a2.q_out_count = cb; a2.q_out_keys = more ? D.keys[side].p : nullptr; a2.unit_counter = ctr + 1;
                            a2.stats = D.stats.p + 1;
                            if (bvh_family) RZ_CUDA(rz_launch_bvh_stage(&a2, (int)p->collect_stats, D.sms, st));
                            else RZ_CUDA(rz_launch_second(&a2, (int)p->collect_stats, D.sms, st));
                            RZ_CUDA(cudaEventRecord(D.stage_ev[2 * ((size_t)pass * n_second + stg) + 1], st));
                            launches += 4;   // count + scan + scatter (rz_sort.cu) + the sorted-segment kernel
                            std::swap(qa, qb); std::swap(ca, cb);
                        }
                        a3.q_in = qa; a3.q_in_count = ca;
                        RZ_CUDA(cudaEventRecord(D.pass_ev[3 * pass + 1], st));
                        a3.unit_counter = ctr + 2;
                        a3.stats = D.stats.p + 2;
                        if (bvh_tail) { a3.set = D.bvhset.view(); a3.self_map = D.brute_to_bvh.p; }
                        if (bvh_family || bvh_tail) RZ_CUDA(rz_launch_bvh(&a3, (int)p->collect_stats, D.sms, st));
                        else RZ_CUDA(rz_launch_path(&a3, ctx->tun.rays_per_thread, (int)p->collect_stats, D.sms, st, nullptr));
                        RZ_CUDA(cudaEventRecord(D.pass_ev[3 * pass + 2], st));
                        launches += 1;
                    }
                    if (n_sides > 1) {   // join the second stream before the resolve
                        RZ_CUDA(cudaEventRecord(D.ev_s2, D.stream2));
                        RZ_CUDA(cudaStreamWaitEvent(D.stream, D.ev_s2, 0));
                    }
                }
            }
        }
        RZ_CUDA(cudaEventRecord(D.ev[2], D.stream));

        RzResolveArgs r;
        r.accum = D.accum.p; r.out_linear = D0.out_linear.p; r.out_rgb8 = D0.out_rgb8.p; r.out_err = nullptr;
        r.n_local_px = n_local; r.width = p->width; r.spp = (uint32_t)next.samples;   // cumulative with RZ_RENDER_ACCUMULATE
        r.dev_index = d; r.dev_count = ND; r.band_rows = band;
        if (host_direct) {   // every device resolves into its OWN compact buffers; rayz_cuda_render copies them out in parallel
            if ((rc = D.loc_linear.alloc((size_t)n_local)) || (rc = D.loc_rgb8.alloc((size_t)n_local * 3))) return rc;
            r.out_linear = D.loc_linear.p; r.out_rgb8 = D.loc_rgb8.p; r.dev_index = 0; r.dev_count = 1;
            D.loc_rows = rows;
        }
        RZ_CUDA(rz_launch_resolve(&r, D.stream));
        if (n_local > 0) launches += 1;
        RZ_CUDA(cudaEventRecord(D.ev[3], D.stream));
        return RZ_OK;
    };
    if (ND == 1) {
        const int rc = per_device(0);
        if (rc) return rc;
    } else {
        std::vector<int> rcs(ND, RZ_OK);
        std::vector<std::string> errs(ND);
        std::vector<std::thread> workers;
        workers.reserve(ND);
        for (uint32_t d = 0; d < ND; d++)
            workers.emplace_back([&, d] { rcs[d] = per_device(d); if (rcs[d]) errs[d] = g_err; });   // g_err is thread-local: hand the text over
        for (std::thread &w : workers) w.join();
        for (uint32_t d = 0; d < ND; d++)
            if (rcs[d]) return rz_fail(rcs[d], "%s", errs[d].c_str());
    }
    uint32_t launches = 0;
    for (uint32_t d = 0; d < ND; d++) launches += launches_dev[d];
    // gather root waits for every peer's resolve (which already wrote into its memory)
    RZ_CUDA(cudaSetDevice(D0.id));
    for (uint32_t d = 1; d < ND; d++) RZ_CUDA(cudaStreamWaitEvent(D0.stream, ctx->devs[d].ev[3], 0));
    RZ_CUDA(cudaEventRecord(D0.ev[4], D0.stream));

    ctx->timing.launches = launches;
    ctx->timing.variant = mega_single ? (uint32_t)RZ_VARIANT_MEGA_SINGLE : variant;
    ctx->stats_valid = false;
    if (sync) {
        for (uint32_t d = 0; d < ND; d++) {
            RZ_CUDA(cudaSetDevice(ctx->devs[d].id));
            RZ_CUDA(cudaStreamSynchronize(ctx->devs[d].stream));
        }
        { const int rc = collect_timing_and_stats(ctx, p->collect_stats != 0); if (rc) return rc; }
        ctx->timing.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_host0).count();
    }
    ctx->acc = next;
    ctx->acc.valid = true;
    ctx->acc.pending = !sync;
    return RZ_OK;
}

// Pre-allocates what a render with these parameters will need (accumulators, result buffers, the staged K1's queues), so
// that the first render does not pay cudaMalloc for ~40 GB: the counterpart of Image.initEmpty in Tracer.init
// (renderer.zig:29-64, image.zig:10-17), which the reference also does before main starts its timer.
extern "C" int rayz_cuda_reserve(RzContext *ctx, const RzRenderParams *p) {
    if (!ctx || !p) return rz_fail(RZ_ERR_INVALID_ARG, "reserve: NULL argument");
    if (p->width == 0 || p->height == 0 || p->spp == 0) return rz_fail(RZ_ERR_INVALID_ARG, "reserve: width, height and spp must be > 0");
    const uint32_t S = p->shard_count <= 1 ? 1 : p->shard_count, s = p->shard_count <= 1 ? 0 : p->shard_index;
    if (s >= S) return rz_fail(RZ_ERR_INVALID_ARG, "reserve: shard_index %u >= shard_count %u", s, S);
    const uint32_t band = p->band_rows ? p->band_rows : 4, ND = (uint32_t)ctx->devs.size();
    if (p->width != ctx->acc.width || p->height != ctx->acc.height || s != ctx->acc.shard_index || S != ctx->acc.shard_count || band != ctx->acc.band_rows)
        ctx->acc.valid = false;   // another frame shape: a next batch may not add to the sums
    DeviceGuard guard;
    int rc;
    Dev &D0 = ctx->devs[0];
    RZ_CUDA(cudaSetDevice(D0.id));
    const uint32_t rows_ctx = rayz_cuda_context_rows(ctx, p->height, p->shard_index, p->shard_count, p->band_rows);
    if ((rc = D0.out_linear.alloc((size_t)rows_ctx * p->width)) || (rc = D0.out_rgb8.alloc((size_t)rows_ctx * p->width * 3))) return rc;
    for (uint32_t d = 0; d < ND; d++) {
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        const uint32_t rows = rayz_cuda_shard_rows(p->height, s * ND + d, S * ND, band);
        const uint32_t n_tiles = (rows * p->width + 31u) / 32u;
        if ((rc = D.accum.alloc((size_t)n_tiles * 32u * 4u)) || (rc = D.counter.alloc(16)) || (rc = D.errword.alloc(4)) || (rc = D.stats.alloc(3))) return rc;
        if (p->variant == RZ_VARIANT_AUTO || p->variant == RZ_VARIANT_MEGA || (p->variant == RZ_VARIANT_BVH && (uint64_t)rows * p->width * p->spp >= (1ull << 26))) {
            const uint32_t chunk = std::min(ctx->tun.chunk_primary, p->spp), n_chunks = (p->spp + chunk - 1) / chunk;
            const uint64_t tiles = std::max<uint64_t>(n_tiles, (uint64_t)((p->width + 7u) / 8u) * ((rows + 3u) / 4u));   // K3's camera stage: 8 x 4 blocks
            if (tiles * n_chunks >= (1ull << 32)) return rz_fail(RZ_ERR_INVALID_ARG, "reserve: too many work units");
            QueuePlan qp;
            if ((rc = plan_and_alloc_queues(ctx->tun, D, qp, (uint32_t)tiles * n_chunks, chunk, (p->flags & RZ_RENDER_SERIAL_PASSES) != 0,
                                            !ctx->have_scene || ctx->n_spheres >= 64u, false, true)))
                return rc;
        }
        RZ_CUDA(cudaStreamSynchronize(D.stream));
    }
    return RZ_OK;
}

extern "C" int rayz_cuda_render_device(RzContext *ctx, const RzCamera *cam, const RzRenderParams *params, void **d_linear_rgba,
                                       void **d_rgb8, uint64_t *out_paths, int sync) {
    const int rc = render_impl(ctx, cam, params, sync != 0);
    if (rc) return rc;
    if (d_linear_rgba) *d_linear_rgba = ctx->devs[0].out_linear.p;
    if (d_rgb8) *d_rgb8 = ctx->devs[0].out_rgb8.p;
    if (out_paths) {
        const uint32_t rows = rayz_cuda_context_rows(ctx, params->height, params->shard_index, params->shard_count, params->band_rows);
        *out_paths = (uint64_t)rows * params->width * params->spp;
    }
    return RZ_OK;
}

// Is this host pointer page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory)?  Only then do async copies from
// several devices run concurrently; pageable memory is staged by the driver one copy at a time.
static bool host_pinned(const void *p) {
    if (!p) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

static int render_host(RzContext *ctx, const RzCamera *cam, const RzRenderParams *params, float *out_linear_rgba, uint8_t *out_rgb8,
                       uint64_t *out_paths);

extern "C" int rayz_cuda_render(RzContext *ctx, const RzCamera *cam, const RzRenderParams *params, float *out_linear_rgba,
                                uint8_t *out_rgb8, uint64_t *out_paths) {
    const int rc = render_host(ctx, cam, params, out_linear_rgba, out_rgb8, out_paths);
    if (ctx) {
        if (rc != RZ_OK && ctx->acc.pending) ctx->acc.valid = false;   // the paths ran but the call failed: the sums are not to be added to
        ctx->acc.pending = false;
    }
    return rc;
}

static int render_host(RzContext *ctx, const RzCamera *cam, const RzRenderParams *params, float *out_linear_rgba, uint8_t *out_rgb8,
                       uint64_t *out_paths) {
    const auto t0 = std::chrono::steady_clock::now();
    if (!ctx || !params) return rz_fail(RZ_ERR_INVALID_ARG, "render: NULL argument");
    // Several devices and page-locked host buffers: no gather to device 0 at all.  Every device resolves its own rows and
    // copies them straight into the caller's frame over its own PCIe link (round 1 funnelled the 157 MB config-3 frame
    // through GPU0's link: 4 % of the step at 8 GPUs).  Rows are dealt in bands, so one strided 2-D copy per device and
    // buffer does it: band lb of device d is rows [(lb * ND + d) * band, ...) of the frame.
    const uint32_t ND = (uint32_t)ctx->devs.size();
    const bool direct = ND > 1 && (out_linear_rgba || out_rgb8) && host_pinned(out_linear_rgba) && host_pinned(out_rgb8);
    const int rc = render_impl(ctx, cam, params, false, direct);
    if (rc) return rc;
    DeviceGuard guard;
    Dev &D0 = ctx->devs[0];
    const uint32_t rows = rayz_cuda_context_rows(ctx, params->height, params->shard_index, params->shard_count, params->band_rows);
    const size_t npx = (size_t)rows * params->width;
    if (direct) {
        const uint32_t band = params->band_rows ? params->band_rows : 4, W = params->width;
        for (uint32_t d = 0; d < ND; d++) {
            Dev &D = ctx->devs[d];
            RZ_CUDA(cudaSetDevice(D.id));
            const uint32_t full = D.loc_rows / band, tail = D.loc_rows - full * band;   // whole bands + a partial last one
            auto copy = [&](void *dst0, const void *src0, size_t px_bytes) -> cudaError_t {
                const size_t band_bytes = (size_t)band * W * px_bytes;
                unsigned char *dst = (unsigned char *)dst0 + (size_t)d * band_bytes;
                cudaError_t e = cudaSuccess;
                if (full) e = cudaMemcpy2DAsync(dst, (size_t)ND * band_bytes, src0, band_bytes, band_bytes, full, cudaMemcpyDeviceToHost, D.stream);
                if (e == cudaSuccess && tail)
                    e = cudaMemcpyAsync(dst + (size_t)full * ND * band_bytes, (const unsigned char *)src0 + (size_t)full * band_bytes, (size_t)tail * W * px_bytes,
                                        cudaMemcpyDeviceToHost, D.stream);
                return e;
            };
            if (out_linear_rgba) RZ_CUDA(copy(out_linear_rgba, D.loc_linear.p, sizeof(float4)));
            if (out_rgb8) RZ_CUDA(copy(out_rgb8, D.loc_rgb8.p, 3));
        }
    } else {
        RZ_CUDA(cudaSetDevice(D0.id));
        if (out_linear_rgba) RZ_CUDA(cudaMemcpyAsync(out_linear_rgba, D0.out_linear.p, npx * sizeof(float4), cudaMemcpyDeviceToHost, D0.stream));
        if (out_rgb8) RZ_CUDA(cudaMemcpyAsync(out_rgb8, D0.out_rgb8.p, npx * 3, cudaMemcpyDeviceToHost, D0.stream));
    }
    for (Dev &D : ctx->devs) {
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaStreamSynchronize(D.stream));
    }
    { const int rc2 = collect_timing_and_stats(ctx, params->collect_stats != 0); if (rc2) return rc2; }
    ctx->timing.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (out_paths) *out_paths = (uint64_t)npx * params->spp;
    return RZ_OK;
}

// Noise of the accumulated frame: every device computes its pixels' errors from its own accumulators with the resolve kernel
// (rows scattered into the gather root's buffer like the image) and reduces them in a fixed order; the host adds the partials
// device by device, CTA by CTA.
extern "C" int rayz_cuda_noise(RzContext *ctx, float target, float *out_err, RzNoise *out) {
    if (!ctx) return rz_fail(RZ_ERR_INVALID_ARG, "noise: ctx is NULL");
    DeviceGuard guard;
    { const int rc = settle_accumulation(ctx); if (rc) return rc; }
    const AccumRecord &A = ctx->acc;
    if (!A.valid) return rz_fail(RZ_ERR_INVALID_ARG, "noise: no accumulated render (none, it failed, or a scene upload or reserve came in between)");
    if (!A.moments) return rz_fail(RZ_ERR_INVALID_ARG, "noise: the accumulated render(s) ran without RZ_RENDER_MOMENTS");
    const uint32_t ND = (uint32_t)ctx->devs.size(), G = rz_noise_grid();
    Dev &D0 = ctx->devs[0];
    const uint32_t rows_ctx = rayz_cuda_context_rows(ctx, A.height, A.shard_index, A.shard_count, A.band_rows);
    int rc;
    RZ_CUDA(cudaSetDevice(D0.id));
    if (out_err && (rc = D0.out_err.alloc((size_t)rows_ctx * A.width))) return rc;
    for (uint32_t d = 0; d < ND; d++) {   // every device enqueues before the first wait
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        const uint32_t n_local = rayz_cuda_shard_rows(A.height, A.shard_index * ND + d, A.shard_count * ND, A.band_rows) * A.width;
        if ((rc = D.noise_part.alloc(4 * (size_t)G))) return rc;
        if (out_err) {
            RzResolveArgs r;
            r.accum = D.accum.p; r.out_linear = nullptr; r.out_rgb8 = nullptr; r.out_err = D0.out_err.p;
            r.n_local_px = n_local; r.width = A.width; r.spp = (uint32_t)A.samples;
            r.dev_index = d; r.dev_count = ND; r.band_rows = A.band_rows;
            RZ_CUDA(rz_launch_resolve(&r, D.stream));
        }
        RZ_CUDA(rz_launch_noise_reduce(D.accum.p, n_local, (uint32_t)A.samples, (double)target, D.noise_part.p, D.stream));
    }
    double sum = 0, sum2 = 0, mx = 0;
    uint64_t above = 0;
    std::vector<double> part(4 * (size_t)G);
    for (Dev &D : ctx->devs) {
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaMemcpyAsync(part.data(), D.noise_part.p, part.size() * sizeof(double), cudaMemcpyDeviceToHost, D.stream));
        RZ_CUDA(cudaStreamSynchronize(D.stream));
        for (uint32_t g = 0; g < G; g++) {
            uint64_t cnt;
            memcpy(&cnt, &part[4 * (size_t)g + 3], sizeof cnt);
            sum += part[4 * (size_t)g]; sum2 += part[4 * (size_t)g + 1]; mx = std::max(mx, part[4 * (size_t)g + 2]); above += cnt;
        }
    }
    if (out_err) {
        RZ_CUDA(cudaSetDevice(D0.id));
        RZ_CUDA(cudaMemcpyAsync(out_err, D0.out_err.p, (size_t)rows_ctx * A.width * sizeof(float), cudaMemcpyDeviceToHost, D0.stream));
        RZ_CUDA(cudaStreamSynchronize(D0.stream));
    }
    if (out) {
        const double npx = (double)rows_ctx * A.width;
        out->samples = A.samples;
        out->n_pixels = rows_ctx * A.width;
        out->n_above = (uint32_t)above;
        out->mean_err = npx > 0 ? sum / npx : 0.0;
        out->rms_err = npx > 0 ? std::sqrt(sum2 / npx) : 0.0;
        out->max_err = mx;
    }
    return RZ_OK;
}

// The stopping policy of progressive rendering, in one place for every host: batches that double the accumulated sample count
// until the frame's rms error reaches the target or max_spp samples are in.
extern "C" int rayz_cuda_render_to_noise(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, float target, uint32_t max_spp,
                                         float *out_linear_rgba, uint8_t *out_rgb8, uint64_t *out_paths, RzNoise *out_noise) {
    const auto t0 = std::chrono::steady_clock::now();
    if (!ctx || !cam || !p) return rz_fail(RZ_ERR_INVALID_ARG, "render_to_noise: NULL argument");
    if (p->spp == 0 || max_spp < p->spp) return rz_fail(RZ_ERR_INVALID_ARG, "render_to_noise: need 0 < spp <= max_spp (spp %u, max_spp %u)", p->spp, max_spp);
    RzRenderParams q = *p;
    q.flags = (p->flags & ~RZ_RENDER_ACCUMULATE) | RZ_RENDER_MOMENTS;
    RzNoise nz;
    memset(&nz, 0, sizeof nz);
    for (;;) {
        int rc = render_impl(ctx, cam, &q, true);
        if (rc) return rc;
        if ((rc = rayz_cuda_noise(ctx, target, nullptr, &nz))) return rc;
        if (nz.rms_err <= (double)target || nz.samples >= max_spp) break;
        q.sample_offset = p->sample_offset + (uint32_t)nz.samples;
        q.spp = (uint32_t)std::min<uint64_t>(nz.samples, max_spp - nz.samples);
        q.flags |= RZ_RENDER_ACCUMULATE;
    }
    DeviceGuard guard;
    Dev &D0 = ctx->devs[0];
    const size_t npx = (size_t)rayz_cuda_context_rows(ctx, p->height, p->shard_index, p->shard_count, p->band_rows) * p->width;
    RZ_CUDA(cudaSetDevice(D0.id));
    if (out_linear_rgba) RZ_CUDA(cudaMemcpyAsync(out_linear_rgba, D0.out_linear.p, npx * sizeof(float4), cudaMemcpyDeviceToHost, D0.stream));
    if (out_rgb8) RZ_CUDA(cudaMemcpyAsync(out_rgb8, D0.out_rgb8.p, npx * 3, cudaMemcpyDeviceToHost, D0.stream));
    RZ_CUDA(cudaStreamSynchronize(D0.stream));
    if (out_paths) *out_paths = (uint64_t)npx * nz.samples;
    if (out_noise) *out_noise = nz;
    ctx->timing.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return RZ_OK;
}

extern "C" int rayz_cuda_primary_ids(RzContext *ctx, const RzCamera *cam, uint32_t width, uint32_t height, int use_bvh,
                                     int32_t *out_ids) {
    if (!ctx || !cam || !out_ids) return rz_fail(RZ_ERR_INVALID_ARG, "primary_ids: NULL argument");
    if (!ctx->have_scene) return rz_fail(RZ_ERR_NO_SCENE, "primary_ids: rayz_cuda_upload_scene has not been called");
    if (width == 0 || height == 0 || (uint64_t)width * height >= (1ull << 31)) return rz_fail(RZ_ERR_INVALID_ARG, "primary_ids: bad image size");
    DeviceGuard guard;
    Dev &D = ctx->devs[0];
    RZ_CUDA(cudaSetDevice(D.id));
    int rc;
    if (use_bvh && !ctx->ref_built) {
        // reference-shaped BVH (hit.zig:130-161), built on first use: O(N log^2 N) on the host
        const uint32_t n = ctx->n_spheres;
        RefBuilder rb;
        rb.h.resize(n);
        for (uint32_t i = 0; i < n; i++) {
            for (int a = 0; a < 3; a++) { rb.h[i].b.lo[a] = ctx->ref_lo[3 * (size_t)i + a]; rb.h[i].b.hi[a] = ctx->ref_hi[3 * (size_t)i + a]; }
            rb.h[i].s = i;
        }
        rb.build(0, n);
        std::vector<uint32_t> reforder(n);
        for (uint32_t i = 0; i < n; i++) reforder[i] = rb.h[i].s;
        if ((rc = D.refnodes.upload(rb.nodes, D.stream))) return rc;
        D.n_refnodes = (uint32_t)rb.nodes.size();
        if ((rc = D.reforder.upload(reforder, D.stream))) return rc;
        RZ_CUDA(cudaStreamSynchronize(D.stream));
        ctx->ref_built = true;
    }
    if ((rc = D.ids.alloc((size_t)width * height))) return rc;
    RzIdsArgs a;
    a.nodes = D.refnodes.p; a.order = D.reforder.p; a.c64 = D.c64_orig.p; a.v64 = D.v64_orig.p;
    a.n_spheres = ctx->n_spheres; a.n_nodes = D.n_refnodes;
    for (int i = 0; i < 3; i++) { a.look_from[i] = cam->look_from[i]; a.px_du[i] = cam->px_du[i]; a.px_dv[i] = cam->px_dv[i]; a.px_origin[i] = cam->px_origin[i]; }
    a.width = width; a.height = height; a.use_bvh = use_bvh; a.out = D.ids.p;
    if ((rc = D.errword.alloc(4))) return rc;
    a.err = D.errword.p;
    RZ_CUDA(cudaMemsetAsync(D.errword.p, 0, 4 * sizeof(unsigned int), D.stream));
    RZ_CUDA(rz_launch_ids(&a, D.stream));
    RZ_CUDA(cudaMemcpyAsync(out_ids, D.ids.p, (size_t)width * height * sizeof(int32_t), cudaMemcpyDeviceToHost, D.stream));
    unsigned int ew = 0;
    RZ_CUDA(cudaMemcpyAsync(&ew, D.errword.p, sizeof ew, cudaMemcpyDeviceToHost, D.stream));
    RZ_CUDA(cudaStreamSynchronize(D.stream));
    if (ew) return rz_fail(RZ_ERR_INTERNAL, "primary_ids: traversal stack overflow (error word 0x%x)", ew);
    return RZ_OK;
}

// Test hook (not in the header): runs the staged K1's key sort (rz_sort.cu) on caller-supplied keys, so that a test can
// check the grouping directly: keys_out ascending, idx_out a permutation of [0, n), keys_in[idx_out[j]] == keys_out[j].
extern "C" int rayz_cuda_debug_sort_keys(RzContext *ctx, const unsigned short *keys, uint32_t n, unsigned short *keys_out, uint32_t *idx_out) {
    if (!ctx || !keys || !keys_out || !idx_out || n == 0 || n > (1u << 28)) return rz_fail(RZ_ERR_INVALID_ARG, "debug_sort_keys: bad argument");
    DeviceGuard guard;
    Dev &D = ctx->devs[0];
    RZ_CUDA(cudaSetDevice(D.id));
    DBuf<unsigned short> ki, ko;
    DBuf<uint32_t> io;
    DBuf<unsigned int> bins, cnt;
    int rc;
    if ((rc = ki.alloc(n)) || (rc = ko.alloc(n)) || (rc = io.alloc(n)) || (rc = bins.alloc(rz_bin_scratch_bytes() / sizeof(unsigned int))) || (rc = cnt.alloc(1))) {
        ki.release(); ko.release(); io.release(); bins.release(); cnt.release();
        return rc;
    }
    cudaError_t e = cudaMemcpyAsync(ki.p, keys, (size_t)n * sizeof(unsigned short), cudaMemcpyHostToDevice, D.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(cnt.p, &n, sizeof n, cudaMemcpyHostToDevice, D.stream);
    if (e == cudaSuccess) e = rz_bin_sort(ki.p, cnt.p, n, bins.p, ko.p, io.p, 1024u, 0u, D.sms, D.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(keys_out, ko.p, (size_t)n * sizeof(unsigned short), cudaMemcpyDeviceToHost, D.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(idx_out, io.p, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, D.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(D.stream);
    ki.release(); ko.release(); io.release(); bins.release(); cnt.release();
    if (e != cudaSuccess) return rz_fail(RZ_ERR_CUDA, "debug_sort_keys: %s", cudaGetErrorString(e));
    return RZ_OK;
}

extern "C" int rayz_cuda_stats(RzContext *ctx, RzStats *out) {
    if (!ctx || !out) return rz_fail(RZ_ERR_INVALID_ARG, "stats: NULL argument");
    if (!ctx->stats_valid) return rz_fail(RZ_ERR_INVALID_ARG, "stats: last render did not run with collect_stats (or was not synchronised)");
    *out = ctx->stats;
    return RZ_OK;
}

extern "C" int rayz_cuda_stage_stats(RzContext *ctx, uint32_t stage, RzStats *out) {
    if (!ctx || !out || stage > 2) return rz_fail(RZ_ERR_INVALID_ARG, "stage_stats: bad argument");
    if (!ctx->stats_valid) return rz_fail(RZ_ERR_INVALID_ARG, "stage_stats: last render did not run with collect_stats (or was not synchronised)");
    *out = ctx->stage_stats[stage];
    return RZ_OK;
}

extern "C" int rayz_cuda_timing(RzContext *ctx, RzTiming *out) {
    if (!ctx || !out) return rz_fail(RZ_ERR_INVALID_ARG, "timing: NULL argument");
    *out = ctx->timing;
    return RZ_OK;
}

extern "C" int rayz_cuda_fp32_peak(RzContext *ctx, uint32_t millis, double *out_tflops, int32_t *out_sms) {
    if (!ctx || !out_tflops) return rz_fail(RZ_ERR_INVALID_ARG, "fp32_peak: NULL argument");
    DeviceGuard guard;
    Dev &D = ctx->devs[0];
    RZ_CUDA(cudaSetDevice(D.id));
    int rc;
    if ((rc = D.sink.alloc(4))) return rc;
    const int grid = D.sms * 8;
    auto run = [&](int iters, int mode, float *ms) -> int {
        RZ_CUDA(cudaEventRecord(D.ev[0], D.stream));
        RZ_CUDA(rz_launch_ffma_peak(D.sink.p, grid, iters, mode, D.stream));
        RZ_CUDA(cudaEventRecord(D.ev[4], D.stream));
        RZ_CUDA(cudaStreamSynchronize(D.stream));
        RZ_CUDA(cudaEventElapsedTime(ms, D.ev[0], D.ev[4]));
        return RZ_OK;
    };
    double best = 0;
    for (int mode = 0; mode < 3; mode++) {   // scalar-operand chains, SGEMM-like 3-register form, packed FFMA2
        float ms = 0;
        if ((rc = run(2000, mode, &ms))) return rc;                 // warm-up
        if ((rc = run(20000, mode, &ms))) return rc;                // calibration
        const double per_iter_ms = ms / 20000.0;
        const int iters = (int)std::min(2.0e9, std::max(1000.0, (millis ? millis : 200) * 0.5 / per_iter_ms));
        if ((rc = run(iters, mode, &ms))) return rc;
        const double flops = 2.0 * 128.0 * (double)iters * 256.0 * (double)grid;
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    *out_tflops = best;
    if (out_sms) *out_sms = D.sms;
    return RZ_OK;
}
