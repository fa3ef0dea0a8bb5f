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
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rayz_cuda.h"
#include "rz_device.cuh"
#include "rz_denoise.cuh"   // RzDenoiseArgs
#include "rz_host_bvh.hpp"   // Box, sphere_box, RefBuilder (K0's reference-shaped BVH), SahBuilder (K3's tree for small scenes)
#include "rz_launch.h"       // the kernel units' launchers and their argument records

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
static const uint32_t RZ_MAX_DEVICES = 8;   // RzConfig::device_ids

// A device allocation that frees itself; whoever destroys one makes its device current (Dev::~Dev).
template <class T>
struct DBuf {
    T *p = nullptr;
    size_t n = 0;
    DBuf() = default;
    DBuf(DBuf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DBuf &operator=(DBuf &&o) noexcept { std::swap(p, o.p); std::swap(n, o.n); return *this; }
    ~DBuf() { release(); }
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
};

struct Dev {
    int id = 0, sms = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t stream2 = nullptr;   // staged K1: odd passes run here so that a pass fills the tail of the previous one
    cudaEvent_t ev_s2 = nullptr, ev_tab = nullptr;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // start, path0, path1, resolve1, done
    SetBufs brute, bvhset;
    DBuf<RzBvhNode> bvh;              // what K3 walks: the builders' binary tree (host SAH or device LBVH), finalized at upload
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
    DBuf<unsigned long long> accum;   // + RZ_RENDER_RQMC's replicate sums and RZ_RENDER_PASSES' pass sums behind the accumulators
                                      // (rz_rep_offset, rz_pass_offset; rz_accum_words)
    DBuf<double> gain;                // RZ_RENDER_RQMC: the segment gains of the local rows (rz_segment_kernel)
    DBuf<double> px_gain;             // RZ_RENDER_RQMC: every local pixel's gain, frozen when an adaptive pixel stops (rz_segment_kernel)
    DBuf<double> pool;                // RZ_RENDER_ADAPTIVE_POOLED: the segment priors U_S of the local rows (rz_segment_kernel)
    DBuf<double> px_pool;             // RZ_RENDER_ADAPTIVE_POOLED: every local pixel's U_S, frozen when it stops (rz_segment_kernel)
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
    DBuf<RzNoisePartial> noise_part;  // rayz_cuda_noise: the reduction's per-CTA partials of this device
    DBuf<uint32_t> out_spp;           // rayz_cuda_pixel_samples: per-pixel sample counts of the context's rows (gather root only)
    DBuf<float4> out_passes;          // rayz_cuda_passes: RZ_PASS_COUNT planes of the context's rows (gather root only)
    DBuf<float4> out_guides;          // rayz_cuda_render_guides: albedo, then normal + depth, of the context's rows (gather root only)
    DBuf<int32_t> out_matte_ids;      // rayz_cuda_render_mattes: [rows * width][ranks] ids and coverage of the context's rows
    DBuf<float> out_matte_cov;        // (gather root only; grown for a larger ranks)
    // rayz_cuda_denoise (gather root only): the resolved frame, then the denoised one; the per-pixel error; the ping-pong pair of
    // (demodulated rgb, variance); the depth gradient; the denoised rgb8.  Never Dev::out_linear / out_rgb8, which a
    // rayz_cuda_render_device caller may still hold.
    DBuf<float4> dn_linear, dn_work;
    DBuf<float> dn_err;
    DBuf<float2> dn_grad;
    DBuf<uint8_t> dn_rgb8;
    DBuf<uint32_t> n_px;              // RZ_RENDER_ADAPTIVE: every local pixel's sample count
    DBuf<uint32_t> px_list;           // RZ_RENDER_ADAPTIVE: the local pixels the next round traces, in increasing order
    DBuf<uint32_t> list_scratch;      // RZ_RENDER_ADAPTIVE: the list kernels' mask words, block offsets and list length (rz_adaptive.cu)
    DBuf<float4> loc_linear;          // multi-device render into HOST buffers: this device's own rows, copied out over its own PCIe link
    DBuf<uint8_t> loc_rgb8;
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

    // With the device current and its streams drained; the DBuf members free themselves after this body.
    ~Dev() {
        if (!own_stream || cudaSetDevice(id) != cudaSuccess) return;   // (own_stream is the first handle rayz_cuda_create makes)
        cudaStreamSynchronize(own_stream);
        if (stream2) cudaStreamSynchronize(stream2);
        if (wf_scratch) rz_wavefront_free(wf_scratch);
        for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : pass_ev) cudaEventDestroy(e);
        for (cudaEvent_t e : stage_ev) cudaEventDestroy(e);
        if (ev_s2) cudaEventDestroy(ev_s2);
        if (ev_tab) cudaEventDestroy(ev_tab);
        if (stream2) cudaStreamDestroy(stream2);
        cudaStreamDestroy(own_stream);
    }
};

// RzRenderParams' image size and shard fields as every render reads them: shard_count 0 or 1 is the whole frame (S = 1,
// s = 0), band_rows 0 means 4.  Equal frames put the same pixels on every device (FrameSplit).
struct Frame {
    uint32_t width = 0, height = 0, S = 1, s = 0, band = 4;
    Frame() = default;
    Frame(uint32_t w, uint32_t h, uint32_t index, uint32_t count, uint32_t band_rows) : width(w), height(h), S(count <= 1 ? 1u : count), s(count <= 1 ? 0u : index), band(band_rows ? band_rows : 4u) {}
    explicit Frame(const RzRenderParams *p) : Frame(p->width, p->height, p->shard_index, p->shard_count, p->band_rows) {}
    bool operator==(const Frame &o) const { return width == o.width && height == o.height && S == o.S && s == o.s && band == o.band; }
    bool operator!=(const Frame &o) const { return !(*this == o); }
};

// What the accumulators of the context's devices hold (RZ_RENDER_ACCUMULATE, include/rayz_cuda.h): the frame and sampling
// parameters a next batch must repeat, and the samples summed so far.  The device set is the context's own.
struct AccumRecord {
    bool valid = false;
    bool pending = false;   // enqueued by rayz_cuda_render_device(sync = 0): the device error words are not checked yet
    Frame frame;
    uint32_t max_depth = 0, moments = 0, sobol = 0, rqmc = 0;
    uint32_t pooled = 0;       // RZ_RENDER_ADAPTIVE_POOLED: every consumer of the error reads the pooled e* (Dev::px_pool)
    uint32_t passes = 0;       // RZ_RENDER_PASSES: the pass sums behind the accumulators hold the frame's light-path passes
    uint32_t filter = 0;       // the flags' pixel-filter field (RZ_RENDER_FILTER), as given
    uint64_t seed = 0;
    float t_min = 0;
    RzCamera cam{};
    uint32_t first_offset = 0;
    uint64_t samples = 0;      // adaptive: the largest per-pixel count (the pixels still active in the last round)
    bool adaptive = false;     // RZ_RENDER_ADAPTIVE: the pixels' counts differ (Dev::n_px), no RZ_RENDER_ACCUMULATE batch continues them
};

// What the gather root's guide buffers (Dev::out_guides) hold after a successful rayz_cuda_render_guides: rayz_cuda_denoise
// takes them for an accumulated frame of the same frame, camera and seed.  A failed guides call, a scene upload or a reserve of
// another frame ends the record, as it ends the accumulation's.
struct GuideRecord {
    bool valid = false;
    Frame frame;
    RzCamera cam{};
    uint64_t seed = 0;
    uint32_t filter = 0;   // the pixel-filter field the guides were traced with (RZ_RENDER_FILTER)
    uint32_t first_offset = 0, samples = 0;
};

struct RzContext {
    explicit RzContext(int n_devices) : devs(n_devices) {}
    std::vector<Dev> devs;
    AccumRecord acc;
    GuideRecord guides;
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

// How a frame is dealt to the context's devices (ctx == nullptr: one device): device d renders shard s * ND + d of S * ND,
// and the gather root's buffers hold the rows of all of them.
struct FrameSplit {
    uint32_t rows[RZ_MAX_DEVICES] = {}, n_local[RZ_MAX_DEVICES] = {};   // per device: rows and pixels
    uint32_t rows_ctx = 0;                                              // of all the devices
    size_t npx = 0;                                                     // pixels of those rows
    FrameSplit() = default;
    FrameSplit(const RzContext *ctx, const Frame &f) {
        const uint32_t nd = ctx ? (uint32_t)ctx->devs.size() : 1u;
        for (uint32_t d = 0; d < nd; d++) {
            rows[d] = rayz_cuda_shard_rows(f.height, f.s * nd + d, f.S * nd, f.band);
            n_local[d] = rows[d] * f.width;
            rows_ctx += rows[d];
        }
        npx = (size_t)rows_ctx * f.width;
    }
};

extern "C" uint32_t rayz_cuda_context_rows(const RzContext *ctx, uint32_t height, uint32_t shard_index, uint32_t shard_count,
                                           uint32_t band_rows) {
    return FrameSplit(ctx, Frame(0, height, shard_index, shard_count, band_rows)).rows_ctx;
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
    if (nd > (int)RZ_MAX_DEVICES) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_create: n_devices %d > %u", nd, RZ_MAX_DEVICES);
    DeviceGuard guard;
    std::unique_ptr<RzContext> ctx(new RzContext(nd));   // an error return tears down what was made so far (Dev::~Dev)
    ctx->flags = cfg ? cfg->flags : 0u;
    ctx->tun = default_tuning();
    for (int d = 0; d < nd; d++) {
        Dev &D = ctx->devs[d];
        D.id = cfg ? cfg->device_ids[d] : 0;
        if (D.id < 0 || D.id >= count) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_create: device id %d out of range (have %d)", D.id, count);
        for (int q = 0; q < d; q++)
            if (ctx->devs[q].id == D.id) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_create: device id %d listed twice", D.id);
    }
    for (int d = 0; d < nd; d++) {
        Dev &D = ctx->devs[d];
        if ((e = cudaSetDevice(D.id)) != cudaSuccess) return rz_fail(RZ_ERR_CUDA, "cudaSetDevice(%d): %s", D.id, cudaGetErrorString(e));
        cudaDeviceProp prop;
        if ((e = cudaGetDeviceProperties(&prop, D.id)) != cudaSuccess) return rz_fail(RZ_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
        if (prop.major < 10) return rz_fail(RZ_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library carries sm_100a code only", D.id, prop.major, prop.minor);
        D.sms = prop.multiProcessorCount;
        if ((e = cudaStreamCreateWithFlags(&D.own_stream, cudaStreamNonBlocking)) != cudaSuccess) return rz_fail(RZ_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        D.stream = D.own_stream;
        if ((e = cudaStreamCreateWithFlags(&D.stream2, cudaStreamNonBlocking)) != cudaSuccess || (e = cudaEventCreateWithFlags(&D.ev_s2, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&D.ev_tab, cudaEventDisableTiming)) != cudaSuccess) return rz_fail(RZ_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        for (auto &ev : D.ev)
            if ((e = cudaEventCreate(&ev)) != cudaSuccess) return rz_fail(RZ_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e));
        if ((e = rz_path_warm()) != cudaSuccess || (e = rz_bvh_warm()) != cudaSuccess || (e = rz_sort_warm()) != cudaSuccess) return rz_fail(RZ_ERR_CUDA, "loading the path kernels: %s", cudaGetErrorString(e));
        if (d > 0) {
            // the resolve kernel of device d stores straight into device 0's buffers (NVLink P2P)
            int can = 0;
            cudaDeviceCanAccessPeer(&can, D.id, ctx->devs[0].id);
            if (!can) return rz_fail(RZ_ERR_UNSUPPORTED, "device %d cannot access peer %d", D.id, ctx->devs[0].id);
            e = cudaDeviceEnablePeerAccess(ctx->devs[0].id, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return rz_fail(RZ_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
            cudaGetLastError();
        }
    }
    *out = ctx.release();
    return RZ_OK;
}

extern "C" void rayz_cuda_destroy(RzContext *ctx) {
    if (!ctx) return;
    DeviceGuard guard;
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

// Runs fn(d) for every device d of the context: inline for one device, else on one host thread PER DEVICE.  ~90 launches per
// pass and device issued from a single thread made device 7 start milliseconds after device 0 (e2e 5 % below the
// device-resident rate at 8 GPUs).  Returns the first failure in device order, with its message.
template <class F>
static int for_each_device(RzContext *ctx, F &&fn) {
    const uint32_t nd = (uint32_t)ctx->devs.size();
    if (nd == 1) return fn(0u);
    int rcs[RZ_MAX_DEVICES] = {};
    std::string errs[RZ_MAX_DEVICES];
    std::thread workers[RZ_MAX_DEVICES];
    for (uint32_t d = 0; d < nd; d++)
        workers[d] = std::thread([&, d] { rcs[d] = fn(d); if (rcs[d]) errs[d] = g_err; });   // g_err is thread-local: hand the text over
    for (uint32_t d = 0; d < nd; d++) workers[d].join();
    for (uint32_t d = 0; d < nd; d++)
        if (rcs[d]) return rz_fail(rcs[d], "%s", errs[d].c_str());
    return RZ_OK;
}

extern "C" int rayz_cuda_upload_scene(RzContext *ctx, const RzScene *sc) {
    if (!ctx || !sc) return rz_fail(RZ_ERR_INVALID_ARG, "rayz_cuda_upload_scene: NULL argument");
    ctx->acc.valid = false;   // sums of the old scene: a next batch may not add to them
    ctx->guides.valid = false;
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
    // one host thread per device (for_each_device): ~25 small copies and allocations each
    auto upload_device = [&](uint32_t d) -> int {
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        int rc;
        if (upload_brute) { if ((rc = upload_set(D.brute, bs, D.stream))) return rc; }
        else { D.brute = SetBufs(); D.brute.n = bs.n; D.brute.n_static = bs.n_static; D.brute.n_static_pad = bs.n_static_pad; D.brute.n_pad = bs.n_pad; }
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
        RZ_CUDA(rz_bvh_finalize(D.bvh.p, D.bvh_nodes, D.stream));   // leaves -> the references K3 follows; no unused slots
        if (device_build) RZ_CUDA(cudaEventRecord(D.ev[1], D.stream));
        if ((rc = D.m_rec.upload(mrec, D.stream)) || (rc = D.m_kind.upload(mk, D.stream)) || (rc = D.m_tex.upload(mt, D.stream)) || (rc = D.m_method.upload(mm, D.stream)) ||
            (rc = D.m_fuzz.upload(mf, D.stream)) || (rc = D.m_ior.upload(mi, D.stream)) || (rc = D.t_kind.upload(tk, D.stream)) ||
            (rc = D.t_even.upload(te, D.stream)) || (rc = D.t_odd.upload(to, D.stream)) || (rc = D.t_color.upload(tc, D.stream)) ||
            (rc = D.t_inv_scale.upload(ts, D.stream)))
            return rc;
        return RZ_OK;
    };
    { const int rc = for_each_device(ctx, upload_device); if (rc) return rc; }
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


// Pass/queue sizing of the staged K1 (see enqueue_staged).
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
    // K3: the tile lists of its camera stage hold 41 KB of shared memory per CTA, and running beside the traversal kernel of the
    // previous pass that stage takes the L1 the kernel's node loads live in (config 4: 247.6 ms overlapped against 212.6 ms in series).
    const bool overlap = !bvh_family;
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

static int sync_devices(RzContext *ctx) {
    for (Dev &D : ctx->devs) {
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaStreamSynchronize(D.stream));
    }
    return RZ_OK;
}

// Every device's error word (RZ_DEV_ERR_*), read behind everything enqueued on its streams: RZ_ERR_INTERNAL if one is set, as
// a device-side capacity was exceeded and work was dropped.  `who` prefixes the message.
static int read_error_words(RzContext *ctx, const char *who = "render") {
    for (Dev &D : ctx->devs) {
        unsigned int ew = 0;
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaMemcpyAsync(&ew, D.errword.p, sizeof ew, cudaMemcpyDeviceToHost, D.stream));
        RZ_CUDA(cudaStreamSynchronize(D.stream));
        if (ew) return rz_fail(RZ_ERR_INTERNAL, "%s: device %d reported%s%s (error word 0x%x): paths were dropped, result withheld", who, D.id,
                               (ew & RZ_DEV_ERR_QUEUE_OVERFLOW) ? " a queue overflow" : "", (ew & RZ_DEV_ERR_STACK_OVERFLOW) ? " a traversal-stack overflow" : "", ew);
    }
    return RZ_OK;
}

// The end of a synchronous render: waits for every device, then reads the device timings (CUDA events), the error words and,
// if asked for, the counters of the render; total_ms is the host time since the caller's t0.
static int finish_render(RzContext *ctx, bool collect_stats, std::chrono::steady_clock::time_point t0) {
    if (const int rc = sync_devices(ctx)) return rc;
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
    if (const int rc = read_error_words(ctx)) return rc;   // the result is not to be used
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
    ctx->timing.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return RZ_OK;
}

// An accumulation left pending by rayz_cuda_render_device(sync = 0): wait for it and read the device error words, so that a
// batch that dropped paths ends the accumulation before anything is added to its sums.
static int settle_accumulation(RzContext *ctx) {
    if (!ctx->acc.valid || !ctx->acc.pending) return RZ_OK;
    ctx->acc.valid = false;
    const int rc = read_error_words(ctx);
    if (rc) return rc == RZ_ERR_INTERNAL ? RZ_OK : rc;   // an error word: stays invalid
    ctx->acc.valid = true;
    ctx->acc.pending = false;
    return RZ_OK;
}

// The accumulated frame, settled, for the readouts of its sums; `who` prefixes the refusal when there is none.
static int accumulated_frame(RzContext *ctx, const char *who, const AccumRecord *&A) {
    if (const int rc = settle_accumulation(ctx)) return rc;
    A = &ctx->acc;
    if (!A->valid) return rz_fail(RZ_ERR_INVALID_ARG, "%s: no accumulated render (none, it failed, or a scene upload or reserve came in between)", who);
    return RZ_OK;
}

// ------------------------------------------------------------------------------ render plan
struct DevPlan {
    uint32_t n_tiles = 0, n_units = 0;                           // n_units: work units of the first kernel
    uint32_t n_list = 0;                                         // adaptive round: the pixels listed on this device
    QueuePlan qp;                                                // staged: the passes alloc_render could allocate
};

// What a render runs and needs, decided before any device is touched: render_impl is plan_render -> alloc_render -> enqueue,
// rayz_cuda_reserve is plan_render -> alloc_render.
struct RenderPlan {
    const RzRenderParams *p = nullptr;
    const RzCamera *cam = nullptr;   // nullptr: planned for rayz_cuda_reserve
    bool host_direct = false;        // every device resolves into its OWN compact buffers; rayz_cuda_render copies them out in parallel
    Frame frame;
    FrameSplit split;
    uint32_t variant = 0;            // resolved to RZ_VARIANT_MEGA, _BVH or _WAVEFRONT
    bool mega_single = false, staged = false;   // staged: enqueue_staged; else one kernel, or the wavefront's own loop
    bool bvh_family = false, bvh_tail = false, enough_spheres = false, serial = false;   // the staged form's plan_queues inputs
    uint32_t chunk = 0, n_chunks = 0, tile_w = 0;   // the first kernel's work-unit size; tile_w: staged K3's camera-stage blocks
    DevPlan dev[RZ_MAX_DEVICES];
    AccumRecord next;                   // what the render commits to ctx->acc when it succeeds
    bool refused = false;               // an RZ_RENDER_ACCUMULATE batch that does not continue `prev`
    bool list = false;                  // an adaptive round after the first: only the pixels of each device's list (Dev::px_list)
};

// Plans a render of these parameters, with the validations (and messages, prefixed `who`) of rayz_cuda_render.  cam == nullptr
// plans for rayz_cuda_reserve: no scene is needed and no accumulation record is made.  n_list (rayz_cuda_render_to_noise's
// adaptive rounds after the first, RZ_RENDER_ADAPTIVE | RZ_RENDER_ACCUMULATE): per device, the length of its pixel list.
// rayz_cuda_render_guides validates its parameters here too and uses the rows of the plan.
static int plan_render(const RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, const AccumRecord &prev, RenderPlan &P,
                       const char *who, const uint32_t *n_list = nullptr) {
    P.p = p;
    P.cam = cam;
    P.list = n_list != nullptr;
    if (cam && !ctx->have_scene) return rz_fail(RZ_ERR_NO_SCENE, "%s: rayz_cuda_upload_scene has not been called", who);
    if (p->width == 0 || p->height == 0 || p->spp == 0) return rz_fail(RZ_ERR_INVALID_ARG, "%s: width, height and spp must be > 0", who);
    if ((uint64_t)p->width * p->height >= (1ull << 31)) return rz_fail(RZ_ERR_INVALID_ARG, "%s: image too large", who);
    P.frame = Frame(p);
    const uint32_t S = P.frame.S, s = P.frame.s, ND = (uint32_t)ctx->devs.size();
    if (s >= S) return rz_fail(RZ_ERR_INVALID_ARG, "%s: shard_index %u >= shard_count %u", who, s, S);
    const Dev &D0 = ctx->devs[0];
    const uint32_t brute_smem = (D0.brute.n_pad * 2 - D0.brute.n_static_pad) * 16u;
    // Every kernel choice looks at the WHOLE FRAME (width x height x spp), never at this shard's or device's share of it: every
    // shard of a frame runs the same kernels, so a sharded render equals the full-frame one bit for bit.
    const uint64_t frame_paths = (uint64_t)p->width * p->height * p->spp;
    P.variant = p->variant;
    if (P.variant == RZ_VARIANT_AUTO) {
        // AUTO picks by cost: the staged brute-force K1 when the sphere set fits shared memory AND the frame is big enough to
        // amortise its ~25 launches per pass (measured one-shot, 485 spheres: 0.9 M paths 3.9 ms vs 0.8 ms for the BVH kernel,
        // 8 M 6.3 vs 2.8, 81 M 23.8 vs 25.3, 405 M 104 vs 125); else the BVH kernel.  (The two kernel families themselves can
        // differ in a pixel or two: FP32 sphere test against exact boxes, tests/test_gpu_parity.py.)
        // An adaptive render runs the BVH family: its rounds after the first are small jobs of scattered pixels.
        P.variant = (p->flags & RZ_RENDER_ADAPTIVE) ? RZ_VARIANT_BVH
                    : (brute_smem <= RZ_SMEM_BUDGET && frame_paths >= (1ull << 26)) ? RZ_VARIANT_MEGA : RZ_VARIANT_BVH;
    }
    // The listed rounds of an adaptive render run the unstaged kernel of the first round's family: K3 for BVH, the single-form
    // K1b for the brute-force family (MEGA, MEGA_SINGLE, WAVEFRONT).  Same family, so every pixel stays exact.
    if (P.list && (P.variant == RZ_VARIANT_MEGA || P.variant == RZ_VARIANT_WAVEFRONT)) P.variant = RZ_VARIANT_MEGA_SINGLE;
    P.mega_single = P.variant == RZ_VARIANT_MEGA_SINGLE;
    if (P.mega_single) P.variant = RZ_VARIANT_MEGA;
    if (P.variant != RZ_VARIANT_MEGA && P.variant != RZ_VARIANT_BVH && P.variant != RZ_VARIANT_WAVEFRONT)
        return rz_fail(RZ_ERR_INVALID_ARG, "%s: unknown variant %u", who, p->variant);
    if (P.variant == RZ_VARIANT_MEGA && brute_smem > RZ_SMEM_BUDGET)
        return rz_fail(RZ_ERR_UNSUPPORTED, "%s: scene needs %u B of shared memory for the brute-force kernel (budget %u); use RZ_VARIANT_BVH", who, brute_smem, RZ_SMEM_BUDGET);
    if (p->flags & RZ_RENDER_RQMC) {   // refused before anything is touched: the accumulated render stays as it was
        const char *rule = !(p->flags & RZ_RENDER_SOBOL) ? "RZ_RENDER_RQMC requires RZ_RENDER_SOBOL"
                           : !(p->flags & RZ_RENDER_MOMENTS) ? "RZ_RENDER_RQMC requires RZ_RENDER_MOMENTS"
                           : (p->spp & 1u) ? "RZ_RENDER_RQMC requires an even spp (two replicates)"
                           : (p->sample_offset & 1u) ? "RZ_RENDER_RQMC requires an even sample_offset (two replicates)" : nullptr;
        if (rule) { P.refused = true; return rz_fail(RZ_ERR_INVALID_ARG, "%s: %s", who, rule); }
    }
    if ((p->flags & RZ_RENDER_ADAPTIVE_POOLED) && !(p->flags & RZ_RENDER_ADAPTIVE)) {
        P.refused = true;
        return rz_fail(RZ_ERR_INVALID_ARG, "%s: RZ_RENDER_ADAPTIVE_POOLED requires RZ_RENDER_ADAPTIVE (rayz_cuda_render_to_noise only)", who);
    }
    {   // the pixel filter's field (RZ_RENDER_FILTER): refused before anything is touched
        const uint32_t kind = rz_filter_kind(p->flags), w16 = (p->flags & RZ_RENDER_FILTER_WIDTH_MASK) >> RZ_RENDER_FILTER_WIDTH_SHIFT;
        if (kind == RZ_FILTER_BOX && w16 != 0u) {
            P.refused = true;
            return rz_fail(RZ_ERR_INVALID_ARG, "%s: RZ_FILTER_BOX takes no width (the width field must be 0; got %u/16 px)", who, w16);
        }
        if (w16 != 0u && (w16 < RZ_FILTER_WIDTH_MIN || w16 > RZ_FILTER_WIDTH_MAX)) {
            P.refused = true;
            return rz_fail(RZ_ERR_INVALID_ARG, "%s: a pixel filter's width must be 0 (the kind's default) or 16..64 sixteenths of a pixel (1 to 4 px; got %u)",
                           who, w16);
        }
    }
    if ((p->flags & RZ_RENDER_PASSES) && p->max_depth > RZ_PASS_MAX_DEPTH) {   // the count must stay out of the kind bits (rz_seg_after_hit)
        P.refused = true;
        return rz_fail(RZ_ERR_INVALID_ARG, "%s: RZ_RENDER_PASSES requires max_depth <= 2^29 - 1 (the first hit's kind rides in the top bits of a path's hit count; got %u)",
                       who, p->max_depth);
    }

    if (cam) {
        AccumRecord &next = P.next;
        next.frame = P.frame;
        next.max_depth = p->max_depth; next.moments = (p->flags & RZ_RENDER_MOMENTS) ? 1u : 0u; next.seed = p->seed;
        next.sobol = (p->flags & RZ_RENDER_SOBOL) ? 1u : 0u;
        next.rqmc = (p->flags & RZ_RENDER_RQMC) ? 1u : 0u;
        next.pooled = (p->flags & RZ_RENDER_ADAPTIVE_POOLED) ? 1u : 0u;
        next.passes = (p->flags & RZ_RENDER_PASSES) ? 1u : 0u;
        next.filter = p->flags & RZ_PATH_FILTER_BITS;
        next.t_min = p->t_min > 0 ? p->t_min : 1e-4f; next.cam = *cam;
        next.first_offset = p->sample_offset; next.samples = p->spp;
        next.adaptive = (p->flags & RZ_RENDER_ADAPTIVE) != 0;
        if (p->flags & RZ_RENDER_ACCUMULATE) {
            auto refuse = [&](const char *why) { P.refused = true; return rz_fail(RZ_ERR_INVALID_ARG, "render: RZ_RENDER_ACCUMULATE refused: %s", why); };
            if (!prev.valid) return refuse("no previous render to add to (none, it failed, or a scene upload or reserve came in between)");
            if (prev.adaptive != next.adaptive)
                return refuse("the accumulated frame was rendered adaptively: its pixels hold different sample counts, so no sample_offset continues it");
            if (prev.frame != next.frame) return refuse("frame size, shard or band_rows differ from the accumulated render");
            if (prev.seed != next.seed || prev.max_depth != next.max_depth || memcmp(&prev.t_min, &next.t_min, sizeof(float)) != 0)
                return refuse("seed, max_depth or t_min differ from the accumulated render");
            if (memcmp(&prev.cam, cam, sizeof(RzCamera)) != 0) return refuse("the camera differs from the accumulated render");
            if (prev.moments != next.moments) return refuse("the RZ_RENDER_MOMENTS bit differs from the accumulated render");
            if (prev.sobol != next.sobol) return refuse("the RZ_RENDER_SOBOL bit differs from the accumulated render");
            if (prev.rqmc != next.rqmc) return refuse("the RZ_RENDER_RQMC bit differs from the accumulated render");
            if (prev.passes != next.passes) return refuse("the RZ_RENDER_PASSES bit differs from the accumulated render");
            if (prev.filter != next.filter) return refuse("the pixel filter (RZ_RENDER_FILTER kind or width) differs from the accumulated render");
            if ((uint64_t)p->sample_offset != (uint64_t)prev.first_offset + prev.samples)
                return refuse("sample_offset must continue where the accumulated samples end (previous sample_offset + spp)");
            if (prev.samples + p->spp > 0xFFFFFFFFull) return refuse("the cumulative sample count would pass 2^32 - 1");
            next.first_offset = prev.first_offset;
            next.samples = prev.samples + p->spp;
        }
    }

    if (P.variant == RZ_VARIANT_BVH) {
        // K3 on a big job: the same staged pipeline with BVH traversal instead of culled lists (sorted rays stay converged); the
        // staged camera stage searches block lists, the unstaged kernel walks the tree
        P.staged = !P.list && ctx->tun.bvh_staged && frame_paths >= (1ull << 26);
    } else if (P.variant == RZ_VARIANT_MEGA) {
        // one persistent kernel for RZ_VARIANT_MEGA_SINGLE, or for a set whose pair lists do not fit beside the primary kernel
        RzPathArgs probe;
        memset(&probe, 0, sizeof probe);
        probe.set = D0.brute.view();
        P.staged = !P.mega_single && rz_primary_smem_bytes(&probe) <= 227u * 1024u;
    }
    if (P.staged) {
        P.bvh_family = P.variant == RZ_VARIANT_BVH;
        // The tail of the paths (whatever survives the sorted stages: incoherent, few) goes to the BVH kernel when the host-built
        // tree is there — ~28 node + sphere tests per segment instead of every sphere of the set (config 2: 29.2 -> 11.1 ms
        // behind four sorted stages).
        P.bvh_tail = !P.bvh_family && D0.brute_to_bvh.p != nullptr && !ctx->tun.tail_brute;
        P.enough_spheres = ctx->n_spheres >= 64u;
        P.serial = (p->flags & RZ_RENDER_SERIAL_PASSES) != 0;
        // The one guess: a reserve before the scene upload cannot know the set, the sphere count or whether there is a BVH tail.
        // It plans the largest staged form (brute force with sorted stages and a BVH tail, both tilings' units); the first
        // render still sizes the sorted stages' pair lists (a function of the set) and, if it runs more passes, their events.
        if (!ctx->have_scene) { P.bvh_family = false; P.bvh_tail = true; P.enough_spheres = true; }
        P.tile_w = P.bvh_family ? 8u : 0u;
    }
    const uint32_t chunk = std::min(ctx->tun.chunk, p->spp), n_chunks = (p->spp + chunk - 1) / chunk;
    P.chunk = P.staged ? std::min(ctx->tun.chunk_primary, p->spp) : chunk;   // the camera-stage kernels build a culled sphere list per unit: their own, larger work-unit size
    P.n_chunks = (p->spp + P.chunk - 1) / P.chunk;
    P.split = FrameSplit(ctx, P.frame);
    for (uint32_t d = 0; d < ND; d++) {
        DevPlan &dp = P.dev[d];
        dp.n_tiles = (P.split.n_local[d] + 31u) / 32u;
        if ((uint64_t)dp.n_tiles * n_chunks >= (1ull << 32)) return rz_fail(RZ_ERR_INVALID_ARG, "%s: too many work units", who);
        uint64_t tiles = dp.n_tiles;
        if (P.list) {   // work unit u: list entries [tile * 32, tile * 32 + 32) x one chunk of samples
            dp.n_list = n_list[d];
            tiles = (dp.n_list + 31u) / 32u;
        }
        const uint64_t blocks = (uint64_t)((p->width + 7u) / 8u) * ((P.split.rows[d] + 3u) / 4u);   // K3's camera stage works on 8 x 4 pixel blocks
        if (P.tile_w) tiles = blocks;
        else if (P.staged && !ctx->have_scene) tiles = std::max(tiles, blocks);
        if (tiles * P.n_chunks >= (1ull << 32)) return rz_fail(RZ_ERR_INVALID_ARG, "%s: too many work units", who);
        dp.n_units = (uint32_t)tiles * P.n_chunks;
    }
    return RZ_OK;
}

// Everything the plan needs on every device, so that enqueueing it allocates nothing.  The one exception is the wavefront
// form's scratch, which rz_wavefront_render sizes itself.
static int alloc_render(RzContext *ctx, RenderPlan &P) {
    int rc;
    if (!P.host_direct) {   // the gather root's frame, into which every device's resolve scatters its rows
        Dev &D0 = ctx->devs[0];
        RZ_CUDA(cudaSetDevice(D0.id));
        if ((rc = D0.out_linear.alloc(P.split.npx)) || (rc = D0.out_rgb8.alloc(P.split.npx * 3))) return rc;
    }
    for (uint32_t d = 0; d < (uint32_t)ctx->devs.size(); d++) {
        Dev &D = ctx->devs[d];
        DevPlan &dp = P.dev[d];
        const uint32_t n_local = P.split.n_local[d];
        RZ_CUDA(cudaSetDevice(D.id));
        const bool rqmc = (P.p->flags & RZ_RENDER_RQMC) != 0;
        const unsigned long long *held = D.accum.p;
        if ((rc = D.accum.alloc(rz_accum_words(dp.n_tiles, rqmc, (P.p->flags & RZ_RENDER_PASSES) != 0)))) return rc;
        if (D.accum.p != held) ctx->acc.valid = false;   // grown (a reserve for RZ_RENDER_RQMC or RZ_RENDER_PASSES of the same frame): the sums are gone
        if (rqmc && ((rc = D.gain.alloc(rz_rqmc_gain_words(n_local, P.frame.width))) || (rc = D.px_gain.alloc(n_local)))) return rc;
        if ((P.p->flags & RZ_RENDER_ADAPTIVE_POOLED) &&
            ((rc = D.pool.alloc(rz_rqmc_gain_words(n_local, P.frame.width))) || (rc = D.px_pool.alloc(n_local))))
            return rc;
        if ((rc = D.counter.alloc(16)) || (rc = D.errword.alloc(4))) return rc;
        if ((rc = D.stats.alloc(3))) return rc;   // [0] whole render / primary kernel, [1] sorted stages, [2] persistent tail kernel
        if (P.staged && n_local > 0) {
            if ((rc = plan_and_alloc_queues(ctx->tun, D, dp.qp, dp.n_units, P.chunk, P.serial, P.enough_spheres, P.bvh_family, P.bvh_tail))) return rc;
            // the sorted-segment kernel's pair lists, one row per sort group
            if (dp.qp.second_stage && !P.bvh_family && ctx->have_scene && (rc = D.bin_lists.alloc((size_t)RZ_SORT_BINS * rz_bin_row_bytes(D.brute.n_pad)))) return rc;
            for (cudaEvent_t e = nullptr; D.pass_ev.size() < 3 * (size_t)dp.qp.n_pass; D.pass_ev.push_back(e)) RZ_CUDA(cudaEventCreate(&e));
            for (cudaEvent_t e = nullptr; D.stage_ev.size() < 2 * (size_t)dp.qp.n_pass * dp.qp.n_second; D.stage_ev.push_back(e)) RZ_CUDA(cudaEventCreate(&e));
        }
        if (P.host_direct && ((rc = D.loc_linear.alloc((size_t)n_local)) || (rc = D.loc_rgb8.alloc((size_t)n_local * 3)))) return rc;
        if ((P.p->flags & RZ_RENDER_ADAPTIVE) &&
            ((rc = D.n_px.alloc(n_local)) || (rc = D.px_list.alloc(n_local)) || (rc = D.list_scratch.alloc(rz_list_scratch_words(n_local)))))
            return rc;
    }
    return RZ_OK;
}

// The staged form on one device: primary kernel (tile-culled camera segments; K3: the block-culled camera stage) -> queue ->
// [sort -> sorted-segment kernel (culled per unit) -> queue] x n_second -> persistent tail kernel (BVH, or brute force).
// Passes are sized by the queues (RzTuning::queue_log2, default 2^27 entries per buffer; two buffers per side, two sides).
// finish_render reads pass_ev and stage_ev by index: their records belong to the streams and places they have here.
static int enqueue_staged(RzContext *ctx, Dev &D, RzPathArgs a, const RenderPlan &P, const QueuePlan &qp, uint32_t &launches) {
    const RzCamera *cam = P.cam;
    const RzRenderParams *p = P.p;
    const int n_sides = qp.n_sides, n_second = qp.n_second;
    const double pcx = cam->px_origin[0] + 0.5 * (p->width - 1) * cam->px_du[0] + 0.5 * (p->height - 1) * cam->px_dv[0] - cam->look_from[0];
    const double pcy = cam->px_origin[1] + 0.5 * (p->width - 1) * cam->px_du[1] + 0.5 * (p->height - 1) * cam->px_dv[1] - cam->look_from[1];
    const double pcz = cam->px_origin[2] + 0.5 * (p->width - 1) * cam->px_du[2] + 0.5 * (p->height - 1) * cam->px_dv[2] - cam->look_from[2];
    a.focus_dist = (float)std::sqrt(pcx * pcx + pcy * pcy + pcz * pcz);   // look_from -> centre of the focus plane
    const double lu = std::sqrt(cam->defocus_u[0] * cam->defocus_u[0] + cam->defocus_u[1] * cam->defocus_u[1] + cam->defocus_u[2] * cam->defocus_u[2]);
    const double lv = std::sqrt(cam->defocus_v[0] * cam->defocus_v[0] + cam->defocus_v[1] * cam->defocus_v[1] + cam->defocus_v[2] * cam->defocus_v[2]);
    a.lens_radius = cam->defocus ? (float)(std::max(lu, lv) * 1.001) : 0.f;
    a.queue_cap = ctx->tun.debug_queue_cap ? std::min((uint32_t)qp.cap, ctx->tun.debug_queue_cap) : (uint32_t)qp.cap;
    rz_key_grid(a, ctx->sb_lo, ctx->sb_hi, ctx->tun.cell_bits, ctx->tun.key_sectors);
    a.huge_radius = ctx->huge_radius;
    uint32_t ue_div = 0;
    if (qp.second_stage && !P.bvh_family) {
        // the sorted-segment kernel's pair lists, one row per sort group: a function of the set and the key grid
        a.bin_row = rz_bin_row_bytes(a.set.n_pad);
        a.bin_lists = D.bin_lists.p;
        RZ_CUDA(rz_launch_bin_lists(&a, D.sms, D.stream));
        launches += 1;
        int grid2 = 0;
        RZ_CUDA(rz_second_grid(&a, (int)p->collect_stats, D.sms, &grid2));
        ue_div = 16u * (uint32_t)grid2;
    }
    RZ_CUDA(cudaEventRecord(D.ev_tab, D.stream));
    D.passes = qp.n_pass;
    D.n_second = (uint32_t)n_second;
    D.queue_entries = (uint32_t)qp.cap;
    D.serial_passes = P.serial;
    // Passes alternate between two streams and two sets of buffers: the persistent kernel ends with a tail of a few long paths
    // (measured ~2 ms per pass), which the next pass's kernels fill.
    if (n_sides > 1) RZ_CUDA(cudaStreamWaitEvent(D.stream2, D.ev_tab, 0));   // (recorded after ev[1] on the same stream)
    uint32_t pass = 0;
    for (uint32_t u0 = 0; u0 < a.n_units; u0 += qp.units_per_pass, pass++) {
        const int side = n_sides > 1 ? (int)(pass & 1u) : 0;
        cudaStream_t st = side ? D.stream2 : D.stream;
        unsigned int *ctr = D.counter.p + 8 * side;   // [0..2] unit counters of K1a/K1c/K1b, [3] entries in q1, [4] entries in q2
        if (pass >= (uint32_t)n_sides) RZ_CUDA(cudaMemsetAsync(ctr, 0, 8 * sizeof(unsigned int), st));
        const uint32_t pass_units = std::min(qp.units_per_pass, a.n_units - u0);
        RzPathArgs a1 = a;
        a1.q_out = D.q1[side].p; a1.q_out_count = ctr + 3; a1.q_out_keys = qp.second_stage ? D.keys[side].p : nullptr;
        a1.unit_base = u0; a1.n_units = pass_units; a1.unit_counter = ctr;
        if (P.bvh_family) RZ_CUDA(rz_launch_bvh_stage(&a1, (int)p->collect_stats, D.sms, st));
        else RZ_CUDA(rz_launch_primary(&a1, (int)p->collect_stats, D.sms, st));
        RZ_CUDA(cudaEventRecord(D.pass_ev[3 * pass], st));
        launches += 1;
        RzPathArgs a3 = a;
        a3.q_in = D.q1[side].p; a3.q_in_count = ctr + 3;
        // sorted, culled stages for the next `n_second` segments: q1 -> q2 -> q1 -> ...
        float4 *qa = D.q1[side].p, *qb = qp.second_stage ? D.q2[side].p : nullptr;
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
            if (P.bvh_family) RZ_CUDA(rz_launch_bvh_stage(&a2, (int)p->collect_stats, D.sms, st));
            else RZ_CUDA(rz_launch_second(&a2, (int)p->collect_stats, D.sms, st));
            RZ_CUDA(cudaEventRecord(D.stage_ev[2 * ((size_t)pass * n_second + stg) + 1], st));
            launches += 4;   // count + scan + scatter (rz_sort.cu) + the sorted-segment kernel
            std::swap(qa, qb); std::swap(ca, cb);
        }
        a3.q_in = qa; a3.q_in_count = ca;
        RZ_CUDA(cudaEventRecord(D.pass_ev[3 * pass + 1], st));
        a3.unit_counter = ctr + 2;
        a3.stats = D.stats.p + 2;
        if (P.bvh_tail) { a3.set = D.bvhset.view(); a3.self_map = D.brute_to_bvh.p; }
        if (P.bvh_family || P.bvh_tail) RZ_CUDA(rz_launch_bvh(&a3, (int)p->collect_stats, D.sms, st));
        else RZ_CUDA(rz_launch_path(&a3, ctx->tun.rays_per_thread, (int)p->collect_stats, D.sms, st, nullptr));
        RZ_CUDA(cudaEventRecord(D.pass_ev[3 * pass + 2], st));
        launches += 1;
    }
    if (n_sides > 1) {   // join the second stream before the resolve
        RZ_CUDA(cudaEventRecord(D.ev_s2, D.stream2));
        RZ_CUDA(cudaStreamWaitEvent(D.stream, D.ev_s2, 0));
    }
    return RZ_OK;
}

// The path-kernel arguments of device d's share of the planned frame that do not depend on the kernel form: the BVH-ordered
// set, scene, camera, frame and shard, sampling (seed, sample range, sampler), t_min, error word and traversal tuning.  rayz_cuda_render_guides launches
// rz_guides_kernel with them as they are (RzGuideArgs); enqueue_device adds the render's buffers and work units.
static RzPathArgs path_args(const RzContext *ctx, const RenderPlan &P, uint32_t d) {
    const RzRenderParams *p = P.p;
    const uint32_t ND = (uint32_t)ctx->devs.size();
    const Dev &D = ctx->devs[d];
    RzPathArgs a;
    memset(&a, 0, sizeof a);
    a.set = D.bvhset.view();
    a.mats.kind = D.m_kind.p; a.mats.fuzz = D.m_fuzz.p; a.mats.ior = D.m_ior.p; a.mats.tex = D.m_tex.p; a.mats.method = D.m_method.p; a.mats.rec = D.m_rec.p;
    a.texs.kind = D.t_kind.p; a.texs.color = D.t_color.p; a.texs.inv_scale = D.t_inv_scale.p; a.texs.even = D.t_even.p; a.texs.odd = D.t_odd.p;
    a.bvh = D.bvh.p; a.bvh_nodes = D.bvh_nodes;
    a.cam = cam_to_f32(P.cam);
    a.width = p->width; a.height = p->height; a.n_local_px = P.split.n_local[d];
    a.spp = p->spp; a.sample_offset = p->sample_offset; a.max_depth = p->max_depth;
    a.shard_index = P.frame.s * ND + d; a.shard_count = P.frame.S * ND; a.band_rows = P.frame.band;
    a.seed_lo = (uint32_t)p->seed; a.seed_hi = (uint32_t)(p->seed >> 32);
    a.sobol = ((p->flags & RZ_RENDER_SOBOL) ? RZ_SAMPLER_SOBOL : 0u) | ((p->flags & RZ_RENDER_RQMC) ? RZ_SAMPLER_RQMC : 0u) |
              ((p->flags & RZ_RENDER_PASSES) ? RZ_PATH_PASSES : 0u) | (p->flags & RZ_PATH_FILTER_BITS);
    a.t_min = P.next.t_min;   // plan_render applied the default
    a.err = D.errword.p;
    a.unit_entries = ctx->tun.unit_entries;
    a.bvh_active_min = (uint32_t)ctx->tun.bvh_active_min; a.bvh_descend_min = (uint32_t)ctx->tun.bvh_descend_min;
    a.stack_cap = ctx->tun.debug_stack_cap;   // 0 = the kernel's own RZ_STACK
    return a;
}

// The resolve kernel's arguments for device d's n_local pixels of the accumulated frame A: its sums, over each pixel's own
// count when A is adaptive, scattered band by band into the gather root's rows.  Every output starts null.  Under RZ_RENDER_RQMC
// and RZ_RENDER_ADAPTIVE_POOLED out_err reads the segment gains and priors, which segment_pass must have enqueued before.
static RzResolveArgs resolve_args(const RzContext *ctx, uint32_t d, const AccumRecord &A, uint32_t n_local) {
    const Dev &D = ctx->devs[d];
    RzResolveArgs r{};
    r.accum = D.accum.p;
    r.n_px = A.adaptive ? D.n_px.p : nullptr;
    r.gain = A.rqmc ? D.px_gain.p : nullptr;
    r.pool = A.pooled ? D.px_pool.p : nullptr;
    r.n_local_px = n_local; r.width = A.frame.width; r.spp = (uint32_t)A.samples;
    r.dev_index = d; r.dev_count = (uint32_t)ctx->devs.size(); r.band_rows = A.frame.band;
    return r;
}

// RZ_RENDER_RQMC and RZ_RENDER_ADAPTIVE_POOLED: device d's segment records of the accumulated frame A, in one launch on its
// stream, before any consumer of the error (the resolve's out_err, the noise reduction, the adaptive flags): the segment gains
// and priors U_S, copied to the pixels whose count is A's largest (every pixel of a uniform frame; the pixels still sampled of an
// adaptive one).  The per-pixel gains and priors those consumers take, or null.
static int segment_pass(RzContext *ctx, uint32_t d, const AccumRecord &A, uint32_t n_local, const double **gain = nullptr,
                        const double **pool = nullptr) {
    Dev &D = ctx->devs[d];
    if (gain) *gain = A.rqmc ? D.px_gain.p : nullptr;
    if (pool) *pool = A.pooled ? D.px_pool.p : nullptr;
    if (!A.rqmc && !A.pooled) return RZ_OK;
    RZ_CUDA(rz_launch_segment_pass(D.accum.p, A.rqmc ? D.accum.p + rz_rep_offset(n_local) : nullptr, A.adaptive ? D.n_px.p : nullptr,
                                   (uint32_t)A.samples, n_local, A.frame.width, A.rqmc ? D.gain.p : nullptr, A.rqmc ? D.px_gain.p : nullptr,
                                   A.pooled ? D.pool.p : nullptr, A.pooled ? D.px_pool.p : nullptr, D.stream));
    return RZ_OK;
}

// Everything device d does for this render, enqueued on its streams into what alloc_render allocated.
static int enqueue_device(RzContext *ctx, const RenderPlan &P, uint32_t d, uint32_t &launches) {
    const RzRenderParams *p = P.p;
    Dev &D = ctx->devs[d], &D0 = ctx->devs[0];
    const DevPlan &dp = P.dev[d];
    const uint32_t n_local = P.split.n_local[d];
    const bool adaptive = (p->flags & RZ_RENDER_ADAPTIVE) != 0;
    const bool trace = n_local > 0 && (!P.list || dp.n_list > 0);   // a device with an empty list launches nothing
    RZ_CUDA(cudaSetDevice(D.id));
    RZ_CUDA(cudaEventRecord(D.ev[0], D.stream));
    if (!(p->flags & RZ_RENDER_ACCUMULATE))   // with the replicate sums and the pass sums behind them under RZ_RENDER_RQMC, RZ_RENDER_PASSES
        RZ_CUDA(cudaMemsetAsync(D.accum.p, 0, rz_accum_words(dp.n_tiles, P.next.rqmc, P.next.passes) * sizeof(unsigned long long), D.stream));
    if (adaptive && !P.list) RZ_CUDA(rz_launch_fill_u32(D.n_px.p, n_local, p->spp, D.stream));   // first round: every pixel
    RZ_CUDA(cudaMemsetAsync(D.counter.p, 0, 16 * sizeof(unsigned int), D.stream));
    RZ_CUDA(cudaMemsetAsync(D.errword.p, 0, 4 * sizeof(unsigned int), D.stream));
    if (p->collect_stats) RZ_CUDA(cudaMemsetAsync(D.stats.p, 0, 3 * sizeof(RzStatsDev), D.stream));

    RzPathArgs a = path_args(ctx, P, d);
    if (P.variant != RZ_VARIANT_BVH) a.set = D.brute.view();
    a.accum = D.accum.p; a.unit_counter = D.counter.p; a.stats = D.stats.p;
    a.chunk = P.chunk; a.n_chunks = P.n_chunks; a.n_units = dp.n_units; a.tile_w = P.tile_w;
    a.moments = P.next.moments;
    if (P.list) { a.px_list = D.px_list.p; a.n_list = dp.n_list; }

    RZ_CUDA(cudaEventRecord(D.ev[1], D.stream));
    D.passes = 0;
    D.n_second = 0;
    D.queue_entries = 0;
    if (trace && P.staged) {
        const int rc = enqueue_staged(ctx, D, a, P, dp.qp, launches);
        if (rc) return rc;
    } else if (trace) {   // one kernel (the wavefront form counts its own launches)
        uint32_t l = 1;
        if (P.variant == RZ_VARIANT_WAVEFRONT) RZ_CUDA(rz_wavefront_render(&a, D.sms, (int)p->collect_stats, D.stream, &D.wf_scratch, &D.wf_scratch_bytes, &l));
        else if (P.variant == RZ_VARIANT_BVH) RZ_CUDA(rz_launch_bvh(&a, (int)p->collect_stats, D.sms, D.stream));
        else RZ_CUDA(rz_launch_path(&a, ctx->tun.rays_per_thread, (int)p->collect_stats, D.sms, D.stream, nullptr));
        launches += l;
    }
    RZ_CUDA(cudaEventRecord(D.ev[2], D.stream));

    RzResolveArgs r = resolve_args(ctx, d, P.next, trace ? n_local : 0u);   // the samples are cumulative with RZ_RENDER_ACCUMULATE
    r.out_linear = D0.out_linear.p; r.out_rgb8 = D0.out_rgb8.p;
    if (P.host_direct) {
        r.out_linear = D.loc_linear.p; r.out_rgb8 = D.loc_rgb8.p; r.dev_index = 0; r.dev_count = 1;
    }
    RZ_CUDA(rz_launch_resolve(&r, D.stream));
    if (trace) launches += 1;
    RZ_CUDA(cudaEventRecord(D.ev[3], D.stream));
    return RZ_OK;
}

static int render_impl(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, bool sync, bool host_direct = false,
                       const uint32_t *n_list = nullptr) {
    if (!ctx || !cam || !p) return rz_fail(RZ_ERR_INVALID_ARG, "render: NULL argument");
    // Every render ends what the accumulators held unless it succeeds (the record is committed at the end) or it is an
    // RZ_RENDER_ACCUMULATE batch that is refused before anything was touched (the record is restored).
    if (p->flags & RZ_RENDER_ACCUMULATE) { DeviceGuard g; const int rc = settle_accumulation(ctx); if (rc) return rc; }
    const AccumRecord prev = ctx->acc;
    ctx->acc.valid = false;
    RenderPlan P;
    if (const int rc = plan_render(ctx, cam, p, prev, P, "render", n_list)) {
        if (P.refused) ctx->acc = prev;
        return rc;
    }
    P.host_direct = host_direct;

    const auto t_host0 = std::chrono::steady_clock::now();
    DeviceGuard guard;
    const uint32_t ND = (uint32_t)ctx->devs.size();
    uint32_t launches_dev[RZ_MAX_DEVICES] = {};
    int rc = alloc_render(ctx, P);
    if (!rc) rc = for_each_device(ctx, [&](uint32_t d) { return enqueue_device(ctx, P, d, launches_dev[d]); });
    if (rc) return rc;
    uint32_t launches = 0;
    for (uint32_t d = 0; d < ND; d++) launches += launches_dev[d];
    // gather root waits for every peer's resolve (which already wrote into its memory)
    Dev &D0 = ctx->devs[0];
    RZ_CUDA(cudaSetDevice(D0.id));
    for (uint32_t d = 1; d < ND; d++) RZ_CUDA(cudaStreamWaitEvent(D0.stream, ctx->devs[d].ev[3], 0));
    RZ_CUDA(cudaEventRecord(D0.ev[4], D0.stream));

    ctx->timing.launches = launches;
    ctx->timing.variant = P.mega_single ? (uint32_t)RZ_VARIANT_MEGA_SINGLE : P.variant;
    ctx->stats_valid = false;
    if (sync && (rc = finish_render(ctx, p->collect_stats != 0, t_host0))) return rc;
    ctx->acc = P.next;
    ctx->acc.valid = true;
    ctx->acc.pending = !sync;
    return RZ_OK;
}

// Pre-allocates what a render with these parameters will need (accumulators, result buffers, the staged K1's queues), so
// that the first render does not pay cudaMalloc for ~40 GB: the counterpart of Image.initEmpty in Tracer.init
// (renderer.zig:29-64, image.zig:10-17), which the reference also does before main starts its timer.  A first render still
// allocates the wavefront scratch, its own rows when several devices render into page-locked host buffers (render_host) and,
// after a reserve made before the scene upload, what plan_render's one guess could not know.
extern "C" int rayz_cuda_reserve(RzContext *ctx, const RzRenderParams *p) {
    if (!ctx || !p) return rz_fail(RZ_ERR_INVALID_ARG, "reserve: NULL argument");
    RenderPlan P;
    int rc = plan_render(ctx, nullptr, p, ctx->acc, P, "reserve");
    if (rc) return rc;
    if (P.frame != ctx->acc.frame) ctx->acc.valid = false;   // another frame shape: a next batch may not add to the sums
    if (P.frame != ctx->guides.frame) ctx->guides.valid = false;
    DeviceGuard guard;
    if ((rc = alloc_render(ctx, P))) return rc;
    return sync_devices(ctx);
}

// RZ_RENDER_ADAPTIVE (and RZ_RENDER_ADAPTIVE_POOLED with it) needs the rounds of rayz_cuda_render_to_noise; a single render
// cannot honour it.
static int refuse_adaptive(const RzRenderParams *p) {
    if (p && (p->flags & RZ_RENDER_ADAPTIVE_POOLED))
        return rz_fail(RZ_ERR_INVALID_ARG, "render: RZ_RENDER_ADAPTIVE_POOLED is honoured by rayz_cuda_render_to_noise with RZ_RENDER_ADAPTIVE only");
    if (p && (p->flags & RZ_RENDER_ADAPTIVE)) return rz_fail(RZ_ERR_INVALID_ARG, "render: RZ_RENDER_ADAPTIVE is honoured by rayz_cuda_render_to_noise only");
    return RZ_OK;
}

extern "C" int rayz_cuda_render_device(RzContext *ctx, const RzCamera *cam, const RzRenderParams *params, void **d_linear_rgba,
                                       void **d_rgb8, uint64_t *out_paths, int sync) {
    if (const int rc = refuse_adaptive(params)) return rc;
    const int rc = render_impl(ctx, cam, params, sync != 0);
    if (rc) return rc;
    if (d_linear_rgba) *d_linear_rgba = ctx->devs[0].out_linear.p;
    if (d_rgb8) *d_rgb8 = ctx->devs[0].out_rgb8.p;
    if (out_paths) *out_paths = (uint64_t)FrameSplit(ctx, Frame(params)).npx * params->spp;
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

// Enqueues the copy of the gathered frame (npx pixels on device 0) into the caller's buffers on device 0's stream.
static int copy_frame_to_host(RzContext *ctx, size_t npx, float *out_linear_rgba, uint8_t *out_rgb8) {
    Dev &D0 = ctx->devs[0];
    RZ_CUDA(cudaSetDevice(D0.id));
    if (out_linear_rgba) RZ_CUDA(cudaMemcpyAsync(out_linear_rgba, D0.out_linear.p, npx * sizeof(float4), cudaMemcpyDeviceToHost, D0.stream));
    if (out_rgb8) RZ_CUDA(cudaMemcpyAsync(out_rgb8, D0.out_rgb8.p, npx * 3, cudaMemcpyDeviceToHost, D0.stream));
    return RZ_OK;
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
    const Frame f(params);
    const FrameSplit sp(ctx, f);
    if (direct) {
        const uint32_t band = f.band, W = f.width;
        for (uint32_t d = 0; d < ND; d++) {
            Dev &D = ctx->devs[d];
            RZ_CUDA(cudaSetDevice(D.id));
            const uint32_t full = sp.rows[d] / band, tail = sp.rows[d] - full * band;   // whole bands + a partial last one
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
        const int rc2 = copy_frame_to_host(ctx, sp.npx, out_linear_rgba, out_rgb8);
        if (rc2) return rc2;
    }
    { const int rc2 = finish_render(ctx, params->collect_stats != 0, t0); if (rc2) return rc2; }
    if (out_paths) *out_paths = (uint64_t)sp.npx * params->spp;
    return RZ_OK;
}

extern "C" int rayz_cuda_render(RzContext *ctx, const RzCamera *cam, const RzRenderParams *params, float *out_linear_rgba,
                                uint8_t *out_rgb8, uint64_t *out_paths) {
    if (const int rc = refuse_adaptive(params)) return rc;
    const int rc = render_host(ctx, cam, params, out_linear_rgba, out_rgb8, out_paths);
    if (ctx) {
        if (rc != RZ_OK && ctx->acc.pending) ctx->acc.valid = false;   // the paths ran but the call failed: the sums are not to be added to
        ctx->acc.pending = false;
    }
    return rc;
}

// Noise of the accumulated frame: every device computes its pixels' errors from its own accumulators with the resolve kernel
// (rows scattered into the gather root's buffer like the image) and reduces them in a fixed order; the host adds the partials
// device by device, CTA by CTA.  An adaptive frame takes each pixel's own sample count.
extern "C" int rayz_cuda_noise(RzContext *ctx, float target, float *out_err, RzNoise *out) {
    if (!ctx) return rz_fail(RZ_ERR_INVALID_ARG, "noise: ctx is NULL");
    DeviceGuard guard;
    const AccumRecord *A = nullptr;
    if (const int rc = accumulated_frame(ctx, "noise", A)) return rc;
    if (!A->moments) return rz_fail(RZ_ERR_INVALID_ARG, "noise: the accumulated render(s) ran without RZ_RENDER_MOMENTS");
    const uint32_t ND = (uint32_t)ctx->devs.size();
    Dev &D0 = ctx->devs[0];
    const FrameSplit sp(ctx, A->frame);
    int rc;
    RZ_CUDA(cudaSetDevice(D0.id));
    if (out_err && (rc = D0.out_err.alloc(sp.npx))) return rc;
    for (uint32_t d = 0; d < ND; d++) {   // every device enqueues before the first wait
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        if ((rc = D.noise_part.alloc(RZ_NOISE_GRID))) return rc;
        const double *gain, *pool;
        if ((rc = segment_pass(ctx, d, *A, sp.n_local[d], &gain, &pool))) return rc;
        if (out_err) {
            RzResolveArgs r = resolve_args(ctx, d, *A, sp.n_local[d]);
            r.out_err = D0.out_err.p;
            RZ_CUDA(rz_launch_resolve(&r, D.stream));
        }
        RZ_CUDA(rz_launch_noise_reduce(D.accum.p, A->adaptive ? D.n_px.p : nullptr, gain, pool, sp.n_local[d], (uint32_t)A->samples,
                                       (double)target, D.noise_part.p, D.stream));
    }
    double sum = 0, sum2 = 0, mx = 0;
    uint64_t above = 0;
    std::vector<RzNoisePartial> part(RZ_NOISE_GRID);
    for (Dev &D : ctx->devs) {
        RZ_CUDA(cudaSetDevice(D.id));
        RZ_CUDA(cudaMemcpyAsync(part.data(), D.noise_part.p, part.size() * sizeof(RzNoisePartial), cudaMemcpyDeviceToHost, D.stream));
        RZ_CUDA(cudaStreamSynchronize(D.stream));
        for (const RzNoisePartial &g : part) { sum += g.sum; sum2 += g.sum2; mx = std::max(mx, g.max); above += g.above; }
    }
    if (out_err) {
        RZ_CUDA(cudaSetDevice(D0.id));
        RZ_CUDA(cudaMemcpyAsync(out_err, D0.out_err.p, sp.npx * sizeof(float), cudaMemcpyDeviceToHost, D0.stream));
        RZ_CUDA(cudaStreamSynchronize(D0.stream));
    }
    if (out) {
        const double npx = (double)sp.npx;
        out->samples = A->samples;
        out->n_pixels = (uint32_t)sp.npx;
        out->n_above = (uint32_t)above;
        out->mean_err = npx > 0 ? sum / npx : 0.0;
        out->rms_err = npx > 0 ? std::sqrt(sum2 / npx) : 0.0;
        out->max_err = mx;
    }
    return RZ_OK;
}

// Per-pixel sample counts of the accumulated frame, laid out like rayz_cuda_noise's out_err: the resolve kernel scatters every
// device's counts (an adaptive frame's own, else the uniform count) into the gather root's buffer.
extern "C" int rayz_cuda_pixel_samples(RzContext *ctx, uint32_t *out_spp) {
    if (!ctx || !out_spp) return rz_fail(RZ_ERR_INVALID_ARG, "pixel_samples: NULL argument");
    DeviceGuard guard;
    const AccumRecord *A = nullptr;
    if (const int rc = accumulated_frame(ctx, "pixel_samples", A)) return rc;
    Dev &D0 = ctx->devs[0];
    const FrameSplit sp(ctx, A->frame);
    int rc;
    RZ_CUDA(cudaSetDevice(D0.id));
    if ((rc = D0.out_spp.alloc(sp.npx))) return rc;
    for (uint32_t d = 0; d < (uint32_t)ctx->devs.size(); d++) {
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        RzResolveArgs r = resolve_args(ctx, d, *A, sp.n_local[d]);
        r.out_spp = D0.out_spp.p;
        RZ_CUDA(rz_launch_resolve(&r, D.stream));
    }
    if ((rc = sync_devices(ctx))) return rc;   // every device's rows are in the gather root's buffer
    RZ_CUDA(cudaSetDevice(D0.id));
    RZ_CUDA(cudaMemcpyAsync(out_spp, D0.out_spp.p, sp.npx * sizeof(uint32_t), cudaMemcpyDeviceToHost, D0.stream));
    RZ_CUDA(cudaStreamSynchronize(D0.stream));
    return RZ_OK;
}

// Light-path passes of the accumulated frame, laid out like rayz_cuda_noise's out_err but RZ_PASS_COUNT planes deep: every
// device's rz_passes_resolve_kernel scatters its rows into the gather root's planes as the resolve does the image.
extern "C" int rayz_cuda_passes(RzContext *ctx, float *out_passes) {
    if (!ctx || !out_passes) return rz_fail(RZ_ERR_INVALID_ARG, "passes: NULL argument");
    DeviceGuard guard;
    const AccumRecord *A = nullptr;
    if (const int rc = accumulated_frame(ctx, "passes", A)) return rc;
    if (!A->passes) return rz_fail(RZ_ERR_INVALID_ARG, "passes: the accumulated render(s) ran without RZ_RENDER_PASSES");
    Dev &D0 = ctx->devs[0];
    const FrameSplit sp(ctx, A->frame);
    int rc;
    RZ_CUDA(cudaSetDevice(D0.id));
    if ((rc = D0.out_passes.alloc((size_t)RZ_PASS_COUNT * sp.npx))) return rc;
    for (uint32_t d = 0; d < (uint32_t)ctx->devs.size(); d++) {
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        const RzResolveArgs r = resolve_args(ctx, d, *A, sp.n_local[d]);
        RZ_CUDA(rz_launch_passes_resolve(&r, D.accum.p + rz_pass_offset(sp.n_local[d], A->rqmc != 0), D0.out_passes.p, sp.npx, D.stream));
    }
    if ((rc = sync_devices(ctx))) return rc;   // every device's rows are in the gather root's planes
    RZ_CUDA(cudaSetDevice(D0.id));
    RZ_CUDA(cudaMemcpyAsync(out_passes, D0.out_passes.p, (size_t)RZ_PASS_COUNT * sp.npx * sizeof(float4), cudaMemcpyDeviceToHost, D0.stream));
    RZ_CUDA(cudaStreamSynchronize(D0.stream));
    return RZ_OK;
}

// Guide buffers (include/rayz_cuda.h): every device traces its rows' camera samples to their first hits with rz_guides_kernel,
// which stores straight into the gather root's buffers like the resolve kernel; the error words are read behind every stream,
// then the root's buffers are copied out.  The accumulators, their record, the per-pixel counts, stats and timing stay as
// they are.
extern "C" int rayz_cuda_render_guides(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, float *out_albedo, float *out_normal) {
    if (!ctx) return rz_fail(RZ_ERR_INVALID_ARG, "guides: NULL argument");
    ctx->guides.valid = false;   // until this call succeeds
    if (!cam || !p) return rz_fail(RZ_ERR_INVALID_ARG, "guides: NULL argument");
    if (p->flags & RZ_RENDER_ADAPTIVE_POOLED)
        return rz_fail(RZ_ERR_INVALID_ARG, "guides: RZ_RENDER_ADAPTIVE_POOLED is honoured by rayz_cuda_render_to_noise with RZ_RENDER_ADAPTIVE only");
    if (p->flags & (RZ_RENDER_ACCUMULATE | RZ_RENDER_ADAPTIVE))
        return rz_fail(RZ_ERR_INVALID_ARG, "guides: RZ_RENDER_ACCUMULATE and RZ_RENDER_ADAPTIVE do not apply to guide buffers");
    if (p->flags & RZ_RENDER_PASSES) return rz_fail(RZ_ERR_INVALID_ARG, "guides: RZ_RENDER_PASSES does not apply to guide buffers");
    RenderPlan P;
    if (const int rc = plan_render(ctx, cam, p, ctx->acc, P, "guides")) return rc;
    DeviceGuard guard;
    // a render enqueued by rayz_cuda_render_device(sync = 0) reports through the error words this call clears: read them first
    { const int rc = settle_accumulation(ctx); if (rc) return rc; }
    const uint32_t ND = (uint32_t)ctx->devs.size();
    const size_t npx = P.split.npx;
    Dev &D0 = ctx->devs[0];
    int rc;
    RZ_CUDA(cudaSetDevice(D0.id));
    if ((rc = D0.out_guides.alloc(2 * npx))) return rc;
    rc = for_each_device(ctx, [&](uint32_t d) -> int {
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        int r;
        if ((r = D.errword.alloc(4))) return r;
        RZ_CUDA(cudaMemsetAsync(D.errword.p, 0, 4 * sizeof(unsigned int), D.stream));
        RzGuideArgs g;
        memset(&g, 0, sizeof g);
        g.a = path_args(ctx, P, d);
        g.out_albedo = D0.out_guides.p;
        g.out_normal = D0.out_guides.p + npx;
        g.dev_index = d; g.dev_count = ND;
        RZ_CUDA(rz_launch_guides(&g, D.stream));
        return RZ_OK;
    });
    if (rc) return rc;
    if ((rc = read_error_words(ctx, "guides"))) return rc;   // behind every device's stream: the root's buffers are complete
    RZ_CUDA(cudaSetDevice(D0.id));
    if (out_albedo) RZ_CUDA(cudaMemcpyAsync(out_albedo, D0.out_guides.p, npx * sizeof(float4), cudaMemcpyDeviceToHost, D0.stream));
    if (out_normal) RZ_CUDA(cudaMemcpyAsync(out_normal, D0.out_guides.p + npx, npx * sizeof(float4), cudaMemcpyDeviceToHost, D0.stream));
    RZ_CUDA(cudaStreamSynchronize(D0.stream));
    GuideRecord &G = ctx->guides;
    G.frame = P.frame; G.cam = *cam; G.seed = p->seed; G.filter = p->flags & RZ_PATH_FILTER_BITS; G.first_offset = p->sample_offset; G.samples = p->spp;
    G.valid = true;
    return RZ_OK;
}

// ID mattes (include/rayz_cuda.h): every device ranks its rows' first-hit ids with rz_mattes_kernel, which stores straight into
// the gather root's buffers as rz_guides_kernel does; the error words are read behind every stream, then the root's buffers
// are copied out.  The accumulators, their record, the per-pixel counts, the guide buffers, stats and timing stay as they are.
extern "C" int rayz_cuda_render_mattes(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, uint32_t ranks,
                                       int32_t *out_ids, float *out_coverage) {
    if (!ctx || !cam || !p) return rz_fail(RZ_ERR_INVALID_ARG, "mattes: NULL argument");
    if (ranks == 0 || ranks > RZ_MATTE_MAX_RANKS) return rz_fail(RZ_ERR_INVALID_ARG, "mattes: ranks %u outside 1..%u", ranks, RZ_MATTE_MAX_RANKS);
    if (p->spp > RZ_MATTE_MAX_SPP) return rz_fail(RZ_ERR_INVALID_ARG, "mattes: spp %u above RZ_MATTE_MAX_SPP (%u)", p->spp, RZ_MATTE_MAX_SPP);
    if (p->flags & (RZ_RENDER_ACCUMULATE | RZ_RENDER_ADAPTIVE | RZ_RENDER_ADAPTIVE_POOLED))
        return rz_fail(RZ_ERR_INVALID_ARG, "mattes: RZ_RENDER_ACCUMULATE, RZ_RENDER_ADAPTIVE and RZ_RENDER_ADAPTIVE_POOLED do not apply to mattes");
    if (p->flags & RZ_RENDER_PASSES) return rz_fail(RZ_ERR_INVALID_ARG, "mattes: RZ_RENDER_PASSES does not apply to mattes");
    RenderPlan P;
    if (const int rc = plan_render(ctx, cam, p, ctx->acc, P, "mattes")) return rc;
    DeviceGuard guard;
    // a render enqueued by rayz_cuda_render_device(sync = 0) reports through the error words this call clears: read them first
    { const int rc = settle_accumulation(ctx); if (rc) return rc; }
    const uint32_t ND = (uint32_t)ctx->devs.size();
    const size_t n = P.split.npx * ranks;
    Dev &D0 = ctx->devs[0];
    int rc;
    RZ_CUDA(cudaSetDevice(D0.id));
    if ((rc = D0.out_matte_ids.alloc(n)) || (rc = D0.out_matte_cov.alloc(n))) return rc;
    rc = for_each_device(ctx, [&](uint32_t d) -> int {
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        int r;
        if ((r = D.errword.alloc(4))) return r;
        RZ_CUDA(cudaMemsetAsync(D.errword.p, 0, 4 * sizeof(unsigned int), D.stream));
        RzMatteArgs g;
        memset(&g, 0, sizeof g);
        g.a = path_args(ctx, P, d);
        g.out_ids = D0.out_matte_ids.p;
        g.out_coverage = D0.out_matte_cov.p;
        g.ranks = ranks;
        g.dev_index = d; g.dev_count = ND;
        RZ_CUDA(rz_launch_mattes(&g, D.stream));
        return RZ_OK;
    });
    if (rc) return rc;
    if ((rc = read_error_words(ctx, "mattes"))) return rc;   // behind every device's stream: the root's buffers are complete
    RZ_CUDA(cudaSetDevice(D0.id));
    if (out_ids) RZ_CUDA(cudaMemcpyAsync(out_ids, D0.out_matte_ids.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, D0.stream));
    if (out_coverage) RZ_CUDA(cudaMemcpyAsync(out_coverage, D0.out_matte_cov.p, n * sizeof(float), cudaMemcpyDeviceToHost, D0.stream));
    RZ_CUDA(cudaStreamSynchronize(D0.stream));
    return RZ_OK;
}

// Denoiser (include/rayz_cuda.h): every device resolves its rows of the accumulated frame (linear and error, or for 0
// iterations linear and rgb8) into the gather root's denoiser buffers, as rayz_cuda_noise does for the error; behind every
// device's stream the root runs rz_denoise.cu alone over the whole frame, so the device count changes no byte.  The
// accumulators, their record, the per-pixel counts, stats, timing and the render's output buffers stay as they are.
extern "C" int rayz_cuda_denoise(RzContext *ctx, const RzDenoiseParams *dp, float *out_linear_rgba, uint8_t *out_rgb8) {
    if (!ctx) return rz_fail(RZ_ERR_INVALID_ARG, "denoise: ctx is NULL");
    RzDenoiseParams q;
    memset(&q, 0, sizeof q);
    q.struct_size = sizeof q;
    q.iterations = 5;
    if (dp) {
        if (dp->struct_size != sizeof(RzDenoiseParams))
            return rz_fail(RZ_ERR_INVALID_ARG, "denoise: struct_size %u != sizeof(RzDenoiseParams) %zu", dp->struct_size, sizeof(RzDenoiseParams));
        if (dp->iterations > 10) return rz_fail(RZ_ERR_INVALID_ARG, "denoise: iterations %u > 10", dp->iterations);
        for (const float s : {dp->sigma_luminance, dp->sigma_normal, dp->sigma_depth})
            if (!(s >= 0.f) || !std::isfinite(s)) return rz_fail(RZ_ERR_INVALID_ARG, "denoise: sigmas must be finite and >= 0 (got %g)", (double)s);
        q = *dp;
    }
    if (q.sigma_luminance == 0.f) q.sigma_luminance = 4.f;
    if (q.sigma_normal == 0.f) q.sigma_normal = 128.f;
    if (q.sigma_depth == 0.f) q.sigma_depth = 1.f;
    DeviceGuard guard;
    const AccumRecord *A = nullptr;
    if (const int rc = accumulated_frame(ctx, "denoise", A)) return rc;
    if (!A->moments) return rz_fail(RZ_ERR_INVALID_ARG, "denoise: the accumulated render(s) ran without RZ_RENDER_MOMENTS: no noise estimate to steer the filter");
    if (A->frame.S > 1)
        return rz_fail(RZ_ERR_UNSUPPORTED, "denoise: the accumulated frame is shard %u of %u: its rows are not image neighbours", A->frame.s, A->frame.S);
    const GuideRecord &G = ctx->guides;
    if (!G.valid)
        return rz_fail(RZ_ERR_INVALID_ARG, "denoise: no guide buffers (none, the last rayz_cuda_render_guides failed, or a scene upload or reserve came in between)");
    if (G.frame != A->frame || memcmp(&G.cam, &A->cam, sizeof(RzCamera)) != 0 || G.seed != A->seed)
        return rz_fail(RZ_ERR_INVALID_ARG, "denoise: the guide buffers' frame, camera or seed differ from the accumulated frame's");
    if (G.filter != A->filter)
        return rz_fail(RZ_ERR_INVALID_ARG, "denoise: the guide buffers' pixel filter (RZ_RENDER_FILTER kind or width) differs from the accumulated frame's");
    const uint32_t ND = (uint32_t)ctx->devs.size();
    Dev &D0 = ctx->devs[0];
    const FrameSplit sp(ctx, A->frame);
    const size_t npx = sp.npx;
    const bool filter = q.iterations > 0;
    int rc;
    RZ_CUDA(cudaSetDevice(D0.id));
    if ((rc = D0.dn_linear.alloc(npx)) || (rc = D0.dn_rgb8.alloc(npx * 3))) return rc;
    if (filter && ((rc = D0.dn_err.alloc(npx)) || (rc = D0.dn_work.alloc(2 * npx)) || (rc = D0.dn_grad.alloc(npx)))) return rc;
    for (uint32_t d = 0; d < ND; d++) {
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        if (filter && (rc = segment_pass(ctx, d, *A, sp.n_local[d]))) return rc;
        RzResolveArgs r = resolve_args(ctx, d, *A, sp.n_local[d]);
        r.out_linear = D0.dn_linear.p;
        if (filter) r.out_err = D0.dn_err.p;
        else r.out_rgb8 = D0.dn_rgb8.p;
        RZ_CUDA(rz_launch_resolve(&r, D.stream));
    }
    if ((rc = sync_devices(ctx))) return rc;   // every device's rows are in the gather root's buffers
    RZ_CUDA(cudaSetDevice(D0.id));
    if (filter) {
        RzDenoiseArgs a;
        memset(&a, 0, sizeof a);
        a.linear = D0.dn_linear.p; a.rgb8 = D0.dn_rgb8.p; a.err = D0.dn_err.p;
        a.albedo = D0.out_guides.p; a.normal = D0.out_guides.p + npx;
        a.work = D0.dn_work.p; a.grad = D0.dn_grad.p;
        a.width = A->frame.width; a.height = A->frame.height; a.iterations = q.iterations;
        a.sigma_l = q.sigma_luminance; a.sigma_n = q.sigma_normal; a.sigma_z = q.sigma_depth;
        RZ_CUDA(rz_launch_denoise(&a, D0.stream));
    }
    if (out_linear_rgba) RZ_CUDA(cudaMemcpyAsync(out_linear_rgba, D0.dn_linear.p, npx * sizeof(float4), cudaMemcpyDeviceToHost, D0.stream));
    if (out_rgb8) RZ_CUDA(cudaMemcpyAsync(out_rgb8, D0.dn_rgb8.p, npx * 3, cudaMemcpyDeviceToHost, D0.stream));
    RZ_CUDA(cudaStreamSynchronize(D0.stream));
    return RZ_OK;
}

// Adaptive rounds: every device lists its active pixels (rz_adaptive.cu: count n_cur, error above the target) and adds `add`
// to their counts; n_list[d] <- the length of device d's list, read behind its stream.
static int build_pixel_lists(RzContext *ctx, uint32_t n_cur, uint32_t add, float target, uint32_t *n_list) {
    const FrameSplit sp(ctx, ctx->acc.frame);
    for (uint32_t d = 0; d < (uint32_t)ctx->devs.size(); d++) {   // every device enqueues before the first wait
        Dev &D = ctx->devs[d];
        RZ_CUDA(cudaSetDevice(D.id));
        const double *gain, *pool;
        if (const int rc = segment_pass(ctx, d, ctx->acc, sp.n_local[d], &gain, &pool)) return rc;
        RZ_CUDA(rz_launch_pixel_list(D.accum.p, gain, pool, D.n_px.p, sp.n_local[d], n_cur, add, target, D.px_list.p,
                                     D.list_scratch.p, D.stream));
        RZ_CUDA(cudaMemcpyAsync(&n_list[d], D.list_scratch.p + rz_list_count_word(sp.n_local[d]), sizeof(uint32_t), cudaMemcpyDeviceToHost, D.stream));
    }
    return sync_devices(ctx);
}

// The stopping policy of progressive rendering, in one place for every host: batches that double the accumulated sample count
// until the frame's rms error reaches the target or max_spp samples are in.  With RZ_RENDER_ADAPTIVE the same schedule runs
// per pixel (DESIGN.md "Adaptive sampling"): after the first round, each round traces only the pixels that took part in every
// earlier round and are still above the target.
extern "C" int rayz_cuda_render_to_noise(RzContext *ctx, const RzCamera *cam, const RzRenderParams *p, float target, uint32_t max_spp,
                                         float *out_linear_rgba, uint8_t *out_rgb8, uint64_t *out_paths, RzNoise *out_noise) {
    const auto t0 = std::chrono::steady_clock::now();
    if (!ctx || !cam || !p) return rz_fail(RZ_ERR_INVALID_ARG, "render_to_noise: NULL argument");
    if (p->spp == 0 || max_spp < p->spp) return rz_fail(RZ_ERR_INVALID_ARG, "render_to_noise: need 0 < spp <= max_spp (spp %u, max_spp %u)", p->spp, max_spp);
    if ((p->flags & RZ_RENDER_RQMC) && (max_spp & 1u))
        return rz_fail(RZ_ERR_INVALID_ARG, "render_to_noise: RZ_RENDER_RQMC requires an even max_spp (two replicates)");
    RzRenderParams q = *p;
    q.flags = (p->flags & ~RZ_RENDER_ACCUMULATE) | RZ_RENDER_MOMENTS;
    RzNoise nz;
    memset(&nz, 0, sizeof nz);
    const size_t npx = FrameSplit(ctx, Frame(p)).npx;
    uint64_t paths = 0;
    if (!(p->flags & RZ_RENDER_ADAPTIVE)) {
        for (;;) {
            int rc = render_impl(ctx, cam, &q, true);
            if (rc) return rc;
            if ((rc = rayz_cuda_noise(ctx, target, nullptr, &nz))) return rc;
            if (nz.rms_err <= (double)target || nz.samples >= max_spp) break;
            q.sample_offset = p->sample_offset + (uint32_t)nz.samples;
            q.spp = (uint32_t)std::min<uint64_t>(nz.samples, max_spp - nz.samples);
            q.flags |= RZ_RENDER_ACCUMULATE;
        }
        paths = (uint64_t)npx * nz.samples;
    } else {
        // Round 0: every pixel, p->spp samples.  Round r + 1: the listed pixels, samples [n, n + b) past sample_offset; a pixel
        // that drops out is never listed again, so every listed pixel holds exactly n samples and all share one sample range.
        int rc = render_impl(ctx, cam, &q, true);
        if (rc) return rc;
        paths = (uint64_t)npx * q.spp;
        q.flags |= RZ_RENDER_ACCUMULATE;
        uint32_t n_list[RZ_MAX_DEVICES] = {};
        for (uint32_t n = p->spp; n < max_spp;) {
            const uint32_t b = std::min(n, max_spp - n);
            {
                DeviceGuard g;
                if ((rc = build_pixel_lists(ctx, n, b, target, n_list))) { ctx->acc.valid = false; return rc; }
            }
            uint64_t listed = 0;
            for (uint32_t d = 0; d < (uint32_t)ctx->devs.size(); d++) listed += n_list[d];
            if (listed == 0) break;
            q.sample_offset = p->sample_offset + n;
            q.spp = b;
            if ((rc = render_impl(ctx, cam, &q, true, false, n_list))) return rc;
            paths += listed * b;
            n += b;
        }
        if ((rc = rayz_cuda_noise(ctx, target, nullptr, &nz))) return rc;
    }
    DeviceGuard guard;
    { const int rc = copy_frame_to_host(ctx, npx, out_linear_rgba, out_rgb8); if (rc) return rc; }
    RZ_CUDA(cudaStreamSynchronize(ctx->devs[0].stream));
    if (out_paths) *out_paths = paths;
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
    if ((rc = ki.alloc(n)) || (rc = ko.alloc(n)) || (rc = io.alloc(n)) || (rc = bins.alloc(rz_bin_scratch_bytes() / sizeof(unsigned int))) || (rc = cnt.alloc(1)))
        return rc;
    cudaError_t e = cudaMemcpyAsync(ki.p, keys, (size_t)n * sizeof(unsigned short), cudaMemcpyHostToDevice, D.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(cnt.p, &n, sizeof n, cudaMemcpyHostToDevice, D.stream);
    if (e == cudaSuccess) e = rz_bin_sort(ki.p, cnt.p, n, bins.p, ko.p, io.p, 1024u, 0u, D.sms, D.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(keys_out, ko.p, (size_t)n * sizeof(unsigned short), cudaMemcpyDeviceToHost, D.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(idx_out, io.p, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, D.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(D.stream);
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
