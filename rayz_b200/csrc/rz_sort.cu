// rz_sort.cu — groups the staged K1's queue entries by the top 12 bits of their sort key (origin cell + direction field):
// a one-pass counting sort written for this job.  Round 1 called cub::DeviceRadixSort here (two 8-bit onesweep passes over
// key + index pairs, ~26 B of HBM traffic per entry, wrapped in a CUDA graph with a SWITCH node because cub wants its item
// count on the host): 12 % of the render step, and a library kernel on the hot path.
//
// What the consumer (rz_second_kernel) needs is weaker than a sort: entries that share (cell, direction) must be contiguous and
// those groups ascending.  The order INSIDE a group is irrelevant — the kernel orders each work unit's entries by the key's
// low 4 bits (the reach class) itself, in shared memory, and radiance is accumulated in integers, so the image does not
// depend on which entries share a work unit.  Without the stability a multi-pass radix sort needs, ONE pass over 4096 bins
// is enough, and 4096 counters fit shared memory:
//   rz_bin_count_kernel    keys -> bins[key >> 4]          per-CTA histogram in shared memory, flushed once   (reads 2 B / entry)
//   rz_bin_scan_kernel     bins -> exclusive prefix = first slot of each group                                (16 KB)
//   rz_bin_scatter_kernel  per tile of 4096 keys: shared-memory histogram gives every key its rank inside (tile, bin); one
//                          global atomicAdd per occupied bin reserves the tile's slots in the group's range; then
//                          idx_out[slot] = entry index | reach class << 28                          (reads 2 B, writes 4 B / entry)
// ~8 B of traffic per entry, no temporary buffers, no global atomic per entry (measured in round 1: +7 ms — the popular
// keys serialise).  The scattered 2- and 4-byte stores land on <= 4096 slowly advancing frontiers that stay in the 126 MB L2
// until their sectors are full.  Every kernel takes the live entry count from device memory: no host round trip, no
// conditional graph, no 0xffff padding keys.
//
// The scan also cuts every group into the consumer's WORK UNITS (at most `ue` consecutive entries of ONE group) and leaves
// their prefix beside the bins: unit_first[b] = units before group b, unit_first[4096] = all units.  A unit never straddles
// two groups, so the consumer knows its rays' cell and direction sector exactly (rz_second_kernel, rz_bin_lists_kernel).
// Scratch layout (unsigned int words, RZ_BIN_* in rz_device.cuh): [0, 4096) bins: counts -> first slot -> (after the
// scatter) END of each group; [4096, 8193) unit_first; [8193] ue, the unit size chosen from the live count.
#include <cuda_runtime.h>
#include <stdint.h>
#include "rz_device.cuh"
#include "rz_launch.h"

namespace {

constexpr int RZ_BINS = RZ_SORT_BINS;                        // 4096 = 12 bits: [origin cell 9][direction 3]
constexpr int RZ_BIN_SHIFT = 4;                              // the key's low 4 bits (reach class) are not sorted on
constexpr int RZ_BIN_THREADS = 256;
constexpr int RZ_BIN_ITEMS = 16;                             // keys per thread and tile
constexpr int RZ_BIN_TILE = RZ_BIN_THREADS * RZ_BIN_ITEMS;   // 4096

struct RzBinArgs {
    const unsigned short *keys_in;   // [n] in producer order
    const unsigned int *count;       // live entries (device counter of the producing kernel)
    uint32_t cap;                    // slots of the buffers (the count is clamped to it)
    unsigned int *bins;              // [4096] counts -> (after the scan) next free slot of each group
    unsigned short *keys_out;        // [n] keys in slot order (null in production: tests only)
    uint32_t *idx_out;               // [n] entry index in slot order | reach class << 28 (RZ_IDX_* in rz_device.cuh)
};

__global__ void __launch_bounds__(RZ_BIN_THREADS) rz_bin_count_kernel(const RzBinArgs a) {
    __shared__ unsigned int sh[RZ_BINS];
    const uint32_t tid = threadIdx.x;
    const uint32_t n = min(*a.count, a.cap);
    for (uint32_t b = tid; b < RZ_BINS; b += RZ_BIN_THREADS) sh[b] = 0u;
    __syncthreads();
    // 8 keys (one 16-byte load) per thread and step; the buffers are 256-byte aligned
    const uint32_t n8 = n >> 3;
    const uint4 *k8 = reinterpret_cast<const uint4 *>(a.keys_in);
    for (uint32_t i = blockIdx.x * RZ_BIN_THREADS + tid; i < n8; i += gridDim.x * RZ_BIN_THREADS) {
        const uint4 v = __ldcs(k8 + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; j++) {
            atomicAdd(&sh[(w[j] & 0xffffu) >> RZ_BIN_SHIFT], 1u);
            atomicAdd(&sh[w[j] >> (16 + RZ_BIN_SHIFT)], 1u);
        }
    }
    if (blockIdx.x == 0 && tid < (n & 7u)) atomicAdd(&sh[(uint32_t)a.keys_in[(n8 << 3) + tid] >> RZ_BIN_SHIFT], 1u);
    __syncthreads();
    for (uint32_t b = tid; b < RZ_BINS; b += RZ_BIN_THREADS) {
        const unsigned int c = sh[b];
        if (c) atomicAdd(a.bins + b, c);
    }
}

// exclusive prefix of 1024 x 4 values held four per thread (one CTA of 1024 threads); returns the thread's own prefix and
// leaves the grand total in *total
__device__ __forceinline__ uint32_t rz_block_prefix(uint32_t sum, uint32_t *s_warp, uint32_t *total) {
    const uint32_t tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    uint32_t inc = sum;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if ((int)lane >= o) inc += t; }
    __syncthreads();   // s_warp may still be read from the previous call
    if (lane == 31u) s_warp[w] = inc;
    __syncthreads();
    if (w == 0u) {
        uint32_t x = s_warp[lane];
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, x, o); if ((int)lane >= o) x += t; }
        s_warp[lane] = x;
    }
    __syncthreads();
    *total = s_warp[31];
    return inc - sum + (w ? s_warp[w - 1u] : 0u);
}

// bins: counts -> first slot of each group (exclusive prefix, in place); unit_first: exclusive prefix of ceil(count / ue) and
// its total; ue = ue_max, but never so many entries that the consumer's warps get fewer than ~4 units each (ue_div = 16 x its
// grid size: the late stages hold a few million entries for 3552 warps).  One CTA, 1024 threads x 4 consecutive bins.
__global__ void __launch_bounds__(1024) rz_bin_scan_kernel(unsigned int *scratch, const unsigned int *count, uint32_t cap, uint32_t ue_max, uint32_t ue_div) {
    __shared__ uint32_t s_warp[32];
    const uint32_t tid = threadIdx.x;
    const uint32_t n = min(*count, cap);
    uint32_t ue = ue_max;
    if (ue > 256u) ue = min(ue, max(256u, (n / max(ue_div, 1u)) & ~63u));
    uint4 *p = reinterpret_cast<uint4 *>(scratch) + tid;
    const uint4 v = *p;
    uint32_t total;
    uint32_t run = rz_block_prefix(v.x + v.y + v.z + v.w, s_warp, &total);
    uint4 o;
    o.x = run; run += v.x;
    o.y = run; run += v.y;
    o.z = run; run += v.z;
    o.w = run;
    *p = o;
    const uint4 u = make_uint4((v.x + ue - 1u) / ue, (v.y + ue - 1u) / ue, (v.z + ue - 1u) / ue, (v.w + ue - 1u) / ue);
    run = rz_block_prefix(u.x + u.y + u.z + u.w, s_warp, &total);
    unsigned int *uf = scratch + RZ_BIN_UNIT_FIRST + 4u * tid;
    uf[0] = run; run += u.x;
    uf[1] = run; run += u.y;
    uf[2] = run; run += u.z;
    uf[3] = run;
    if (tid == 0u) { scratch[RZ_BIN_UNIT_FIRST + RZ_SORT_BINS] = total; scratch[RZ_BIN_UE] = ue; }
}

__global__ void __launch_bounds__(RZ_BIN_THREADS) rz_bin_scatter_kernel(const RzBinArgs a) {
    __shared__ unsigned int sh[RZ_BINS];   // entries of the bin in this tile; after the reservation: their first global slot
    const uint32_t tid = threadIdx.x;
    const uint32_t n = min(*a.count, a.cap);
    const uint32_t n_tiles = (n + RZ_BIN_TILE - 1) / RZ_BIN_TILE;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (uint32_t b = tid; b < RZ_BINS; b += RZ_BIN_THREADS) sh[b] = 0u;
        __syncthreads();
        const uint32_t i0 = tile * RZ_BIN_TILE + tid;
        uint32_t key[RZ_BIN_ITEMS], rank[RZ_BIN_ITEMS];
#pragma unroll
        for (int j = 0; j < RZ_BIN_ITEMS; j++) {
            const uint32_t i = i0 + (uint32_t)j * RZ_BIN_THREADS;
            key[j] = i < n ? (uint32_t)a.keys_in[i] : 0xffffffffu;
        }
#pragma unroll
        for (int j = 0; j < RZ_BIN_ITEMS; j++) rank[j] = key[j] != 0xffffffffu ? atomicAdd(&sh[key[j] >> RZ_BIN_SHIFT], 1u) : 0u;
        __syncthreads();
        for (uint32_t b = tid; b < RZ_BINS; b += RZ_BIN_THREADS) {
            const unsigned int c = sh[b];
            if (c) sh[b] = atomicAdd(a.bins + b, c);   // the tile's slots in the group's range
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < RZ_BIN_ITEMS; j++) {
            if (key[j] != 0xffffffffu) {
                const uint32_t pos = sh[key[j] >> RZ_BIN_SHIFT] + rank[j];
                if (pos < a.cap) {   // always true: the ranges partition [0, n)
                    // entry index (< 2^28: RzTuning::queue_log2 <= 28) with the key's reach class in the top four bits: the
                    // consumer needs nothing else of the key, and a second scattered 2-byte store per entry is the expensive kind
                    a.idx_out[pos] = (i0 + (uint32_t)j * RZ_BIN_THREADS) | ((key[j] & 15u) << 28);
                    if (a.keys_out) a.keys_out[pos] = (unsigned short)key[j];   // tests only
                }
            }
        }
        __syncthreads();
    }
}

}  // namespace

extern "C" size_t rz_bin_scratch_bytes(void) { return (size_t)RZ_BIN_SCRATCH_WORDS * sizeof(unsigned int); }

// keys_in[0, *count) -> idx_out (/ keys_out when not null): entry indices (+ class bits) and keys grouped by ascending (key >> 4).  bins: rz_bin_scratch_bytes()
// (layout above).  ue_max, ue_div: work-unit size of the consumer and 16 x its grid size.
extern "C" cudaError_t rz_bin_sort(const unsigned short *keys_in, const unsigned int *count, uint32_t cap, unsigned int *bins,
                                   unsigned short *keys_out, uint32_t *idx_out, uint32_t ue_max, uint32_t ue_div, int sm_count, cudaStream_t stream) {
    // resident CTAs per SM of the two kernels (called from one host thread per device: no shared mutable state here)
    int per_sm_count = 0, per_sm_scatter = 0;
    cudaError_t eo = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_count, rz_bin_count_kernel, RZ_BIN_THREADS, 0);
    if (eo == cudaSuccess) eo = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_scatter, rz_bin_scatter_kernel, RZ_BIN_THREADS, 0);
    if (eo != cudaSuccess) return eo;
    if (per_sm_count < 1 || per_sm_scatter < 1) return cudaErrorInvalidConfiguration;
    RzBinArgs a;
    a.keys_in = keys_in; a.count = count; a.cap = cap; a.bins = bins; a.keys_out = keys_out; a.idx_out = idx_out;
    const unsigned tiles = (cap + RZ_BIN_TILE - 1) / RZ_BIN_TILE;
    auto grid_for = [&](int per_sm) { const unsigned g = (unsigned)(sm_count * per_sm); return tiles < g ? (tiles ? tiles : 1u) : g; };
    cudaError_t e = cudaMemsetAsync(bins, 0, (size_t)RZ_BINS * sizeof(unsigned int), stream);
    if (e != cudaSuccess) return e;
    rz_bin_count_kernel<<<grid_for(per_sm_count), RZ_BIN_THREADS, 0, stream>>>(a);
    rz_bin_scan_kernel<<<1, 1024, 0, stream>>>(bins, count, cap, ue_max ? ue_max : 1024u, ue_div);
    rz_bin_scatter_kernel<<<grid_for(per_sm_scatter), RZ_BIN_THREADS, 0, stream>>>(a);
    return cudaGetLastError();
}

extern "C" cudaError_t rz_sort_warm(void) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, rz_bin_count_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, rz_bin_scatter_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, rz_bin_scan_kernel);
    return e;
}
