// rz_adaptive.cu — the pixel lists of adaptive sampling (RZ_RENDER_ADAPTIVE, DESIGN.md "Adaptive sampling").
//
// Before each round after the first, a pixel stays active iff it took part in every earlier round (its count is the current
// N) and its error is above the target: the same float comparison rz_noise_reduce_kernel makes for n_above.  The active
// pixels of a device are written in increasing local index by a scan, not an atomic append, so that consecutive list
// entries are neighbouring pixels and a warp's camera rays stay coherent.  Three small kernels over the device's pixels:
//   flag    : one 32-bit mask word per warp of 32 pixels, and the count of each block of RZ_LIST_BLOCK pixels;
//   scan    : one CTA turns the block counts into block offsets and writes the list length;
//   scatter : every active pixel goes to its place in the list, and its count grows by the round's batch.
#include "rz_device.cuh"   // rz_pixel_err_of
#include "rz_launch.h"

#define RZ_LIST_BLOCK 1024u   // pixels (one per thread) per block of the flag and scatter kernels

// gain, pool (nullable): RZ_RENDER_RQMC's per-pixel gains and RZ_RENDER_ADAPTIVE_POOLED's priors, as rz_noise_reduce_kernel takes them.
__global__ void __launch_bounds__(RZ_LIST_BLOCK) rz_list_flag_kernel(const unsigned long long *__restrict__ accum,
                                                                     const double *__restrict__ gain, const double *__restrict__ pool,
                                                                     const uint32_t *__restrict__ n_px, uint32_t n_local_px,
                                                                     uint32_t n_cur, double target, uint32_t *__restrict__ mask,
                                                                     uint32_t *__restrict__ block_count) {
    __shared__ uint32_t s_cnt[32];
    const uint32_t lp = blockIdx.x * RZ_LIST_BLOCK + threadIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    bool active = false;
    if (lp < n_local_px && n_px[lp] == n_cur) {
        const unsigned long long *q = accum + (size_t)lp * 4;
        active = (double)(float)rz_pixel_err_of(q, n_cur, gain, pool, lp) > target;
    }
    const uint32_t m = __ballot_sync(0xffffffffu, active);
    if (lane == 0) {
        mask[(size_t)blockIdx.x * 32u + warp] = m;
        s_cnt[warp] = __popc(m);
    }
    __syncthreads();
    if (warp == 0) {
        uint32_t c = s_cnt[lane];
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0) block_count[blockIdx.x] = c;
    }
}

// block_count -> exclusive offsets in place; *total = the list length.  One CTA, 1024 blocks per step.
__global__ void __launch_bounds__(1024) rz_list_scan_kernel(uint32_t *__restrict__ block_count, uint32_t n_blocks, uint32_t *__restrict__ total) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_blocks; base += 1024u) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < n_blocks ? block_count[i] : 0u;
        uint32_t x = v;   // inclusive scan within the warp
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (uint32_t)o) x += y;
        }
        if (lane == 31u) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {   // inclusive scan of the warp totals
            uint32_t w = s_warp[lane];
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= (uint32_t)o) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        if (i < n_blocks) block_count[i] = s_carry + (warp ? s_warp[warp - 1] : 0u) + x - v;
        __syncthreads();
        if (threadIdx.x == 0) s_carry += s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = s_carry;
}

__global__ void __launch_bounds__(RZ_LIST_BLOCK) rz_list_scatter_kernel(const uint32_t *__restrict__ mask, const uint32_t *__restrict__ block_offset,
                                                                        uint32_t n_local_px, uint32_t add, uint32_t *__restrict__ n_px,
                                                                        uint32_t *__restrict__ list) {
    __shared__ uint32_t s_off[32];
    const uint32_t lp = blockIdx.x * RZ_LIST_BLOCK + threadIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t *bm = mask + (size_t)blockIdx.x * 32u;
    if (warp == 0) {   // exclusive offsets of the block's 32 warps
        const uint32_t c = __popc(bm[lane]);
        uint32_t x = c;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (uint32_t)o) x += y;
        }
        s_off[lane] = x - c;
    }
    __syncthreads();
    const uint32_t m = bm[warp];
    if (lp < n_local_px && ((m >> lane) & 1u)) {
        list[block_offset[blockIdx.x] + s_off[warp] + __popc(m & ((1u << lane) - 1u))] = lp;
        n_px[lp] += add;
    }
}

__global__ void __launch_bounds__(256) rz_fill_u32_kernel(uint32_t *__restrict__ p, uint32_t n, uint32_t v) {
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    if (i < n) p[i] = v;
}

static uint32_t rz_list_blocks(uint32_t n_local_px) { return (n_local_px + RZ_LIST_BLOCK - 1u) / RZ_LIST_BLOCK; }

// Scratch of rz_launch_pixel_list, in words: the mask words, the block offsets, then the list length (at rz_list_count_word).
extern "C" size_t rz_list_scratch_words(uint32_t n_local_px) { return (size_t)rz_list_blocks(n_local_px) * 33u + 1u; }
extern "C" size_t rz_list_count_word(uint32_t n_local_px) { return (size_t)rz_list_blocks(n_local_px) * 33u; }

// The active pixels of this device before the next round: list <- every local pixel with n_px == n_cur and error > target,
// in increasing order; their counts grow by `add`; scratch[rz_list_count_word(n_local_px)] <- the list length.  gain, pool
// (nullable): RZ_RENDER_RQMC's per-pixel gains and RZ_RENDER_ADAPTIVE_POOLED's priors, so that the error is the one
// rayz_cuda_noise shows.
extern "C" cudaError_t rz_launch_pixel_list(const unsigned long long *accum, const double *gain, const double *pool, uint32_t *n_px,
                                            uint32_t n_local_px, uint32_t n_cur, uint32_t add,
                                            float target, uint32_t *list, uint32_t *scratch, cudaStream_t stream) {
    const uint32_t nb = rz_list_blocks(n_local_px);
    uint32_t *mask = scratch, *block = scratch + (size_t)nb * 32u, *total = scratch + rz_list_count_word(n_local_px);
    if (nb) rz_list_flag_kernel<<<nb, RZ_LIST_BLOCK, 0, stream>>>(accum, gain, pool, n_px, n_local_px, n_cur, (double)target, mask, block);
    rz_list_scan_kernel<<<1, 1024, 0, stream>>>(block, nb, total);
    if (nb) rz_list_scatter_kernel<<<nb, RZ_LIST_BLOCK, 0, stream>>>(mask, block, n_local_px, add, n_px, list);
    return cudaGetLastError();
}

// Every local pixel's count <- v (the first round of an adaptive render).
extern "C" cudaError_t rz_launch_fill_u32(uint32_t *p, uint32_t n, uint32_t v, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    rz_fill_u32_kernel<<<(n + 255u) / 256u, 256, 0, stream>>>(p, n, v);
    return cudaGetLastError();
}
