// rz_sampler.cuh — the low-discrepancy sampler of RZ_RENDER_SOBOL (include/rayz_cuda.h, DESIGN.md "Low-discrepancy sampling").
// RZ_HD so that tests/hostsim/sampler.cu compiles the same code as host code and tests/test_sampler_cpu.py compares it with an
// independent numpy restatement.
//
// Each pixel draws its uniforms in 2-D pairs, every pair an Owen-scrambled Sobol (0,2)-sequence with its own padding (Burley 2020,
// "Practical Hash-based Owen Scrambling", JCGT 9(4)):
//   S(x, s)     = brev(LK(brev(x), s))            nested-uniform scramble; LK = Laine-Karras-style hash (rz_lk_hash)
//   i'          = S(i, seed of the shuffle)       shuffled sample index: aligned blocks of 2^k indices stay aligned blocks
//   point i     = (S(D0(i'), seed x), S(D1(i'), seed y))
//   D0(i)       = brev(i)                         Sobol dimension 0 (van der Corput)
//   D1(i)       = XOR over the set bits j of i of V_j, V_j = m_j << (31 - j), m_0 = 1, m_j = m_{j-1} ^ (m_{j-1} << 1)
//                                                 Sobol dimension 1 (Joe-Kuo d = 2: s = 1, a = 0, m = {1})
// The seeds are rz_hash32 chains of (seed, global pixel, pair) only (rz_sobol_pair_seed): never of the sample index.
// Included by rz_device.cuh, after RZ_HD and rz_u01.
#pragma once

// Pairs: camera A (jitter x, y), camera B (lens radius, angle), camera C (shutter time, first coordinate only), then bounce
// s = 1..max_depth (the scatter's u.x, u.y) as pair 2 + s.
enum { RZ_PAIR_CAMERA_JITTER = 0, RZ_PAIR_CAMERA_LENS = 1, RZ_PAIR_CAMERA_TIME = 2 };
RZ_HD uint32_t rz_pair_bounce(uint32_t s) { return 2u + s; }

RZ_HD uint32_t rz_brev(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __brev(x);
#else
    x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
    x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
    x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
    x = ((x >> 8) & 0x00FF00FFu) | ((x & 0x00FF00FFu) << 8);
    return (x >> 16) | (x << 16);
#endif
}

// lowbias32 (C. Wellons, "Prospecting for hash functions", 2018): a bijective 32-bit mixer
RZ_HD uint32_t rz_hash32(uint32_t x) {
    x ^= x >> 16;
    x *= 0x7feb352du;
    x ^= x >> 15;
    x *= 0x846ca68bu;
    x ^= x >> 16;
    return x;
}

// Burley's Laine-Karras-style permutation: bit b of the result depends on bits <= b of x only (each step adds or XORs a
// multiple of x by an even constant), and it is a bijection.  Applied between two bit reversals it is an Owen scramble.
RZ_HD uint32_t rz_lk_hash(uint32_t x, uint32_t seed) {
    x += seed;
    x ^= x * 0x6c50b47cu;
    x ^= x * 0xb82f1e52u;
    x ^= x * 0xc7afe638u;
    x ^= x * 0x8d22f6e6u;
    return x;
}

RZ_HD uint32_t rz_owen_scramble(uint32_t x, uint32_t seed) { return rz_brev(rz_lk_hash(rz_brev(x), seed)); }

RZ_HD uint32_t rz_sobol_d0(uint32_t i) { return rz_brev(i); }

// Sobol dimension 1.  Its generator matrix is Pascal's triangle mod 2 (m_j = row j), so bit k of brev(D1(i)) is the XOR of the bits
// n of i with C(n, k) odd, i.e. with k a subset of n (Lucas): a superset-sum transform, five shift-mask steps instead of 32.
RZ_HD uint32_t rz_sobol_d1(uint32_t i) {
    i ^= (i >> 1) & 0x55555555u;
    i ^= (i >> 2) & 0x33333333u;
    i ^= (i >> 4) & 0x0F0F0F0Fu;
    i ^= (i >> 8) & 0x00FF00FFu;
    i ^= i >> 16;
    return rz_brev(i);
}

// Base seed of one pair of one pixel; the shuffle and the two coordinate scrambles take rz_hash32(base ^ 0), (base ^ 1), (base ^ 2).
RZ_HD uint32_t rz_sobol_pair_seed(uint32_t k0, uint32_t k1, uint32_t gpix, uint32_t pair) {
    uint32_t h = rz_hash32(k0 ^ 0x6a09e667u);
    h = rz_hash32(h ^ k1);
    h = rz_hash32(h ^ gpix);
    return rz_hash32(h ^ pair);
}

// RZ_RENDER_RQMC: the base seed of replicate r (0 or 1) of a pair, from the pair's own base seed
RZ_HD uint32_t rz_rqmc_replicate_seed(uint32_t base, uint32_t r) { return rz_hash32(base ^ (0x9e3779b9u + r)); }

// The 32-bit coordinates of sample `sample` of `pair` for pixel gpix (callers keep the top 24 bits: rz_u01(x >> 8)).
// `rqmc` (RZ_RENDER_RQMC): sample i is sample i >> 1 of replicate i & 1, a sequence of its own (rz_rqmc_replicate_seed).
RZ_HD uint2 rz_sobol_pair(uint32_t k0, uint32_t k1, uint32_t gpix, uint32_t pair, uint32_t sample, bool rqmc = false) {
    uint32_t base = rz_sobol_pair_seed(k0, k1, gpix, pair);
    if (rqmc) {
        base = rz_rqmc_replicate_seed(base, sample & 1u);
        sample >>= 1;
    }
    const uint32_t i = rz_owen_scramble(sample, rz_hash32(base));
    return make_uint2(rz_owen_scramble(rz_sobol_d0(i), rz_hash32(base ^ 1u)), rz_owen_scramble(rz_sobol_d1(i), rz_hash32(base ^ 2u)));
}

// The pair's two uniforms: rz_u01 of the top 24 bits of each coordinate.
RZ_HD float2 rz_sobol_u01(uint32_t k0, uint32_t k1, uint32_t gpix, uint32_t pair, uint32_t sample, bool rqmc = false) {
    const uint2 q = rz_sobol_pair(k0, k1, gpix, pair, sample, rqmc);
    return make_float2(rz_u01(q.x >> 8), rz_u01(q.y >> 8));
}
