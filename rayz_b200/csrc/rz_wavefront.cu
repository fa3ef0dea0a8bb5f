// rz_wavefront.cu — K2: the staged ("wavefront") variant of the path tracer, the comparison
// point for the megakernel (BASELINE.json north_star: "compared against a wavefront variant that
// uses warp-ballot compaction by material and by terminated path").
//
// A pool of M path slots lives in HBM as structure-of-arrays.  One iteration =
//   generate : refill free slots with the next (pixel, sample) paths           (camera.zig:59-77)
//   intersect: closest hit for every live slot (shared-memory brute force, as K1), then each
//              slot index is appended to the queue of its outcome — miss / diffuse / metallic /
//              dielectric — with warp-ballot compaction (__ballot_sync + __popc, one atomic
//              per warp per queue)
//   shade    : one warp = 32 entries of ONE queue (queues start on 32-entry boundaries), so the
//              material switch of Material.scatter (material.zig:167-176) is warp-uniform;
//              survivors are compacted into the next live list, terminated paths into the free
//              list, again by ballot
//   advance  : one thread swaps the lists and resets the counters
// Eight iterations are captured once into a CUDA graph and replayed until the device-side
// `done` flag is set; the host reads the flag once per replay.
// The same search/shade device functions as the megakernel are used (rz_search.cuh) and the
// RNG is keyed by (pixel, sample, bounce), so both variants produce bit-identical images.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "rz_launch.h"
#include "rz_search.cuh"

struct WfCounters {
    unsigned int n_live;       // entries of live[cur]
    unsigned int n_next;       // entries being appended to live[cur ^ 1] by shade
    unsigned int n_free;       // entries of the free list (a stack)
    unsigned int q_count[4];   // miss, diffuse, metallic, dielectric
    unsigned int q_off[4];     // queue starts inside `queue`, 32-aligned
    unsigned int q_total;      // padded total
    unsigned int cur;          // which live list is current
    unsigned int n_gen;        // paths generated in this iteration
    unsigned int done;
    unsigned int pad;
    unsigned long long next_path;   // next global path index to start
    unsigned long long total_paths;
};

struct WfState {
    float4 *A;   // ox oy oz time
    float4 *B;   // dx dy dz self_k(bits)
    float4 *C;   // thr.rgb seg(bits)
    uint4 *D;    // lp gpix sample bk
    unsigned int *live[2];
    unsigned int *free_list;
    unsigned int *queue;      // 4 queues, capacity M + 128 in total
    WfCounters *ctr;
    RzStatsDev *stats;
    unsigned int M;
};

__global__ void wf_init(WfState s, unsigned long long total_paths) {
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < s.M) s.free_list[i] = s.M - 1u - i;
    if (i == 0) {
        WfCounters c;
        memset(&c, 0, sizeof c);
        c.n_free = s.M;
        c.total_paths = total_paths;
        *s.ctr = c;
    }
}

// path index g -> (local pixel, sample): tile-major like the megakernel's work units
__device__ __forceinline__ void wf_decode(const RzPathArgs &a, unsigned long long g, uint32_t &lp, uint32_t &sample) {
    const unsigned long long per_tile = 32ull * a.spp;
    const uint32_t tile = (uint32_t)(g / per_tile);
    const uint32_t r = (uint32_t)(g - (unsigned long long)tile * per_tile);
    lp = tile * 32u + (r & 31u);
    sample = r >> 5;
}

template <bool STATS, int SOBOL, bool FILTER = false>
__global__ void __launch_bounds__(256) wf_generate(const RzPathArgs a, WfState s) {
    const WfCounters c = *s.ctr;
    const unsigned long long remaining = c.total_paths - c.next_path;
    const unsigned int n_new = (unsigned int)min((unsigned long long)c.n_free, remaining);
    unsigned long long c_paths = 0, c_depth = 0;
    for (unsigned int t = blockIdx.x * blockDim.x + threadIdx.x; t < n_new; t += gridDim.x * blockDim.x) {
        const unsigned int slot = s.free_list[c.n_free - 1u - t];
        uint32_t lp, sample;
        wf_decode(a, c.next_path + t, lp, sample);
        uint4 d = make_uint4(lp, 0u, a.sample_offset + sample, 0xffffffffu);
        float4 A = make_float4(0.f, 0.f, 0.f, 0.f), B = make_float4(0.f, 1.f, 0.f, __int_as_float(-1));
        float4 C = make_float4(0.f, 0.f, 0.f, __uint_as_float(0u));
        bool alive = false;
        if (lp < a.n_local_px) {
            uint32_t pi, pj;
            rz_local_to_global(lp, a.width, a.shard_index, a.shard_count, a.band_rows, pi, pj);
            d.y = pj * a.width + pi;
            const RzRay ray = rz_camera_ray(a.cam, pi, pj, d.y, d.z, a.seed_lo, a.seed_hi, SOBOL, FILTER ? a.sobol : 0u);
            A = make_float4(ray.o.x, ray.o.y, ray.o.z, ray.time);
            B = make_float4(ray.d.x, ray.d.y, ray.d.z, __int_as_float(ray.self_k));
            C = make_float4(1.f, 1.f, 1.f, __uint_as_float(0u));
            alive = a.max_depth > 0u;
            if (STATS) { c_paths++; if (!alive) c_depth++; }
        }
        s.A[slot] = A; s.B[slot] = B; s.C[slot] = C; s.D[slot] = d;
        // dead-on-arrival paths (padding pixels, max_depth 0) are marked by thr = 0 and an
        // infinitely distant origin is not needed: they go through one miss with zero radiance
        if (!alive) s.C[slot] = make_float4(0.f, 0.f, 0.f, __uint_as_float(0x80000000u));
        s.live[c.cur][c.n_live + t] = slot;
    }
    if (STATS) {
        for (int o = 16; o > 0; o >>= 1) { c_paths += __shfl_xor_sync(0xffffffffu, c_paths, o); c_depth += __shfl_xor_sync(0xffffffffu, c_depth, o); }
        if ((threadIdx.x & 31u) == 0) { if (c_paths) atomicAdd(&s.stats->v[0], c_paths); if (c_depth) atomicAdd(&s.stats->v[9], c_depth); }
    }
}

__global__ void wf_after_generate(WfState s) {
    WfCounters *c = s.ctr;
    const unsigned long long remaining = c->total_paths - c->next_path;
    const unsigned int n_new = (unsigned int)min((unsigned long long)c->n_free, remaining);
    c->n_free -= n_new;
    c->n_live += n_new;
    c->next_path += n_new;
    c->n_gen = n_new;
    for (int q = 0; q < 4; q++) c->q_count[q] = 0;
    // queue regions sized for the worst case: every live path in one queue
    c->n_next = 0;
}

// warp-ballot compaction: append `slot` of every lane with `flag` to list[*counter ...]
__device__ __forceinline__ void wf_push(bool flag, unsigned int slot, unsigned int *list, unsigned int *counter) {
    const unsigned mask = __ballot_sync(0xffffffffu, flag);
    if (mask == 0u) return;
    const unsigned lane = threadIdx.x & 31u;
    unsigned int base = 0;
    if (lane == (unsigned)(__ffs(mask) - 1)) base = atomicAdd(counter, (unsigned int)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, __ffs(mask) - 1);
    if (flag) list[base + __popc(mask & ((1u << lane) - 1u))] = slot;
}

template <int R>
__global__ void __launch_bounds__(128) wf_intersect(const RzPathArgs a, WfState s) {
    extern __shared__ __align__(16) unsigned char rz_smem[];
    __shared__ __align__(8) uint64_t s_bar;
    float4 *s_pk = reinterpret_cast<float4 *>(rz_smem);
    rz_stage_scene_pk(a.set, s_pk, &s_bar);
    const WfCounters c = *s.ctr;
    const unsigned int n = c.n_live;
    const unsigned int *live = s.live[c.cur];
    const unsigned int M = s.M;
    // each of the 4 queues owns a region of M+32 entries: no overflow whatever the split
    const unsigned int stride = gridDim.x * blockDim.x;
    const unsigned int n_round = (n + R * 32u - 1u) / (R * 32u) * (R * 32u);
    for (unsigned int t0 = (blockIdx.x * blockDim.x + threadIdx.x); t0 * R < n_round; t0 += stride) {
        // a warp covers R*32 consecutive entries: lane handles entries base + lane + 32*r
        const unsigned int warp_base = (t0 & ~31u) * R;
        const unsigned int lane = t0 & 31u;
        RzRay rays[R];
        unsigned int slot[R];
        bool valid[R];
        float bt[R];
        int bk[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            const unsigned int e = warp_base + lane + 32u * r;
            valid[r] = e < n;
            slot[r] = valid[r] ? live[e] : 0u;
            const float4 A = valid[r] ? s.A[slot[r]] : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 B = valid[r] ? s.B[slot[r]] : make_float4(0.f, 1.f, 0.f, __int_as_float(-1));
            rays[r].o = f3(A.x, A.y, A.z); rays[r].time = A.w;
            rays[r].d = f3(B.x, B.y, B.z); rays[r].self_k = __float_as_int(B.w);
            bt[r] = 3.0e38f; bk[r] = -1;
        }
        rz_search_brute2<R, 2>(s_pk, (int)a.set.n_static_pad, (int)a.set.n_pad, rays, a.t_min, bt, bk);
#pragma unroll
        for (int r = 0; r < R; r++) {
            unsigned int q = 4u;
            if (valid[r]) {
                // dead-on-arrival marker: force a (zero-radiance) miss
                const bool doa = (__float_as_uint(s.C[slot[r]].w) & 0x80000000u) != 0u;
                if (doa) bk[r] = -1;
                s.D[slot[r]].w = (unsigned int)bk[r];
                q = 0u;
                if (bk[r] >= 0) q = 1u + min(a.mats.kind[a.set.mat[bk[r] & ~RZ_FAR_BIT]], 2u);
            }
#pragma unroll
            for (unsigned int qq = 0; qq < 4u; qq++)
                wf_push(q == qq, slot[r], s.queue + (size_t)qq * (M + 32u), &s.ctr->q_count[qq]);
        }
    }
}

__global__ void wf_after_intersect(WfState s) {
    WfCounters *c = s.ctr;
    unsigned int off = 0;
    for (int q = 0; q < 4; q++) {
        c->q_off[q] = off;
        off += (c->q_count[q] + 31u) & ~31u;
    }
    c->q_total = off;
}

template <bool STATS, int SOBOL, bool PASSES>
__global__ void __launch_bounds__(256) wf_shade(const RzPathArgs a, WfState s) {
    const WfCounters c = *s.ctr;
    const unsigned int M = s.M;
    unsigned int *next_live = s.live[c.cur ^ 1u];
    unsigned long long c_segs = 0, c_hit[3] = {0, 0, 0}, c_sky = 0, c_abs = 0, c_depth = 0;
    for (unsigned int t = blockIdx.x * blockDim.x + threadIdx.x; t < c.q_total; t += gridDim.x * blockDim.x) {
        // warp-uniform queue lookup: queue starts are multiples of 32
        unsigned int q = 3u;
        if (t < c.q_off[1]) q = 0u; else if (t < c.q_off[2]) q = 1u; else if (t < c.q_off[3]) q = 2u;
        const unsigned int e = t - c.q_off[q];
        const bool valid = e < c.q_count[q];
        bool survive = false, died = false;
        unsigned int slot = 0;
        if (valid) {
            slot = s.queue[(size_t)q * (M + 32u) + e];
            const float4 A = s.A[slot], B = s.B[slot], C = s.C[slot];
            const uint4 D = s.D[slot];
            RzRay ray;
            ray.o = f3(A.x, A.y, A.z); ray.time = A.w; ray.d = f3(B.x, B.y, B.z); ray.self_k = __float_as_int(B.w);
            float3 thr = f3(C.x, C.y, C.z);
            const bool doa = (__float_as_uint(C.w) & 0x80000000u) != 0u;
            uint32_t seg = __float_as_uint(C.w) & 0x7fffffffu;
            uint32_t kind;
            int res;
            if (doa) { res = RZ_END_DEPTH; kind = 3u; }
            else {
                if (STATS) c_segs++;
                res = rz_shade_segment(a, ray, thr, seg, D.x, D.y, D.z, (int)D.w, kind, SOBOL, PASSES);
                if (STATS) {
                    if (kind < 3u) c_hit[kind]++;
                    if (res == RZ_END_SKY) c_sky++;
                    if (res == RZ_END_ABSORBED) c_abs++;
                    if (res == RZ_END_DEPTH) c_depth++;
                }
            }
            if (res == RZ_CONT) {
                s.A[slot] = make_float4(ray.o.x, ray.o.y, ray.o.z, ray.time);
                s.B[slot] = make_float4(ray.d.x, ray.d.y, ray.d.z, __int_as_float(ray.self_k));
                s.C[slot] = make_float4(thr.x, thr.y, thr.z, __uint_as_float(seg));
                survive = true;
            } else {
                died = true;
            }
        }
        wf_push(survive, slot, next_live, &s.ctr->n_next);
        wf_push(died, slot, s.free_list, &s.ctr->n_free);
    }
    if (STATS) {
        unsigned long long v[7] = {c_segs, c_hit[0], c_hit[1], c_hit[2], c_sky, c_abs, c_depth};
        const int idx[7] = {1, 4, 5, 6, 7, 8, 9};
#pragma unroll
        for (int i = 0; i < 7; i++) {
            unsigned long long x = v[i];
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            if ((threadIdx.x & 31u) == 0 && x) atomicAdd(&s.stats->v[idx[i]], x);
        }
    }
}

__global__ void wf_advance(WfState s) {
    WfCounters *c = s.ctr;
    c->cur ^= 1u;
    c->n_live = c->n_next;
    c->n_next = 0;
    c->done = (c->n_live == 0u && c->next_path >= c->total_paths) ? 1u : 0u;
}

// ------------------------------------------------------------------------------ host driver
struct WfScratch {
    WfState st;
    cudaGraphExec_t graph[2];   // [stats]
    RzPathArgs captured[2];
    bool have_graph[2];
    unsigned int *h_done;       // pinned
    size_t M;
};

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

extern "C" cudaError_t rz_wavefront_render(const RzPathArgs *a, int sm_count, int collect_stats, cudaStream_t stream,
                                           void **scratch, size_t *scratch_bytes, uint32_t *launches) {
    cudaError_t e;
    const unsigned long long n_tiles = (a->n_local_px + 31u) / 32u;
    const unsigned long long total_paths = n_tiles * 32ull * a->spp;   // padding pixels are dead on arrival
    const int pool_log2 = 21;   // 2^21 slots: 2^21..2^25 measured within 10 % of each other (DESIGN.md section 5)
    const size_t M = (size_t)std::min<unsigned long long>(total_paths, 1ull << pool_log2);
    WfScratch *ws = reinterpret_cast<WfScratch *>(*scratch);
    if (!ws || ws->M < M) {
        if (ws) {
            for (int i = 0; i < 2; i++) if (ws->have_graph[i]) cudaGraphExecDestroy(ws->graph[i]);
            cudaFree(ws->st.A); cudaFreeHost(ws->h_done); delete ws;
        }
        ws = new WfScratch();
        memset(ws, 0, sizeof *ws);
        ws->M = M;
        // one slab: A,B,C,D (16 B each per slot), live x2, free, queue x4(+32), counters
        const size_t bytes = align256(M * 16) * 4 + align256(M * 4) * 3 + align256((M + 32) * 4 * 4) + 256;
        unsigned char *base = nullptr;
        if ((e = cudaMalloc((void **)&base, bytes)) != cudaSuccess) { delete ws; *scratch = nullptr; return e; }
        size_t off = 0;
        auto take = [&](size_t n) { unsigned char *p = base + off; off += align256(n); return p; };
        ws->st.A = (float4 *)take(M * 16); ws->st.B = (float4 *)take(M * 16); ws->st.C = (float4 *)take(M * 16); ws->st.D = (uint4 *)take(M * 16);
        ws->st.live[0] = (unsigned int *)take(M * 4); ws->st.live[1] = (unsigned int *)take(M * 4); ws->st.free_list = (unsigned int *)take(M * 4);
        ws->st.queue = (unsigned int *)take((M + 32) * 4 * 4);
        ws->st.ctr = (WfCounters *)take(256);
        ws->st.M = (unsigned int)M;
        if ((e = cudaMallocHost((void **)&ws->h_done, sizeof(unsigned int))) != cudaSuccess) { cudaFree(base); delete ws; *scratch = nullptr; return e; }
        *scratch = ws;
        *scratch_bytes = bytes;
    }
    ws->st.stats = a->stats;
    const int st = collect_stats ? 1 : 0;
    const size_t smem = (size_t)(a->set.n_pad + (a->set.n_pad - a->set.n_static_pad)) * 16u;
    const int grid_i = sm_count * 8, grid_s = sm_count * 4;
    uint32_t n_launch = 0;
    // the pool may be larger than this job needs (scratch reused after a bigger render): the free list is rebuilt over ALL
    // of its ws->M slots, or the stale top of the stack would hand out slots the rewritten bottom also holds
    wf_init<<<(unsigned)((ws->M + 255) / 256), 256, 0, stream>>>(ws->st, total_paths);
    n_launch++;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;

    // (re)capture the 8-iteration graph when the arguments change (kernel params are baked in)
    const int ITERS = 8;
    if (!ws->have_graph[st] || memcmp(&ws->captured[st], a, sizeof *a) != 0) {
        if (ws->have_graph[st]) { cudaGraphExecDestroy(ws->graph[st]); ws->have_graph[st] = false; }
        if ((e = cudaFuncSetAttribute(wf_intersect<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        cudaStream_t cap;
        if ((e = cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking)) != cudaSuccess) return e;
        cudaGraph_t g;
        if ((e = cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal)) != cudaSuccess) return e;
        for (int it = 0; it < ITERS; it++) {
            rz_pick_camera_instance(*a, st, [](auto S, auto M, auto, auto F) { return wf_generate<decltype(S)::value, decltype(M)::value, decltype(F)::value>; })<<<grid_s, 256, 0, cap>>>(*a, ws->st);
            wf_after_generate<<<1, 1, 0, cap>>>(ws->st);
            wf_intersect<2><<<grid_i, 128, smem, cap>>>(*a, ws->st);
            wf_after_intersect<<<1, 1, 0, cap>>>(ws->st);
            rz_pick_instance(*a, st, [](auto S, auto M, auto P) { return wf_shade<decltype(S)::value, decltype(M)::value, decltype(P)::value>; })<<<grid_s, 256, 0, cap>>>(*a, ws->st);
            wf_advance<<<1, 1, 0, cap>>>(ws->st);
        }
        cudaMemcpyAsync(ws->h_done, &ws->st.ctr->done, sizeof(unsigned int), cudaMemcpyDeviceToHost, cap);
        if ((e = cudaStreamEndCapture(cap, &g)) != cudaSuccess) { cudaStreamDestroy(cap); return e; }
        e = cudaGraphInstantiate(&ws->graph[st], g, 0);
        cudaGraphDestroy(g);
        cudaStreamDestroy(cap);
        if (e != cudaSuccess) return e;
        ws->captured[st] = *a;
        ws->have_graph[st] = true;
    }
    // replay until the device says every path has terminated
    const unsigned long long segs_bound = total_paths * (unsigned long long)std::max(1u, a->max_depth) / M + 64ull;
    for (unsigned long long rep = 0; rep < segs_bound + 8; rep++) {
        *ws->h_done = 0;
        if ((e = cudaGraphLaunch(ws->graph[st], stream)) != cudaSuccess) return e;
        n_launch += ITERS * 6;
        if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
        if (*ws->h_done) break;
    }
    if (launches) *launches = n_launch;
    return cudaSuccess;
}

extern "C" void rz_wavefront_free(void *scratch) {
    WfScratch *ws = reinterpret_cast<WfScratch *>(scratch);
    if (!ws) return;
    for (int i = 0; i < 2; i++) if (ws->have_graph[i]) cudaGraphExecDestroy(ws->graph[i]);
    cudaFree(ws->st.A);
    cudaFreeHost(ws->h_done);
    delete ws;
}
