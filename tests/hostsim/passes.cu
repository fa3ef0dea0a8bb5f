// Test-only: the light-path pass rule of RZ_RENDER_PASSES (rz_device.cuh's rz_pass_of and the seg word's encoding,
// rz_seg_after_hit / rz_seg_hits / rz_seg_first_kind) compiled as HOST code, so that tests/test_passes_cpu.py can check it
// against a table.  The product only ever runs these functions inside its CUDA kernels.
#include <cstdint>

#include "../../rayz_b200/csrc/rz_device.cuh"

extern "C" uint32_t hostpass_count(void) { return RZ_PASS_COUNT; }
extern "C" uint32_t hostpass_max_depth(void) { return RZ_PASS_MAX_DEPTH; }
extern "C" uint32_t hostpass_of(uint32_t hits, uint32_t first_kind) { return rz_pass_of(hits, first_kind); }
extern "C" uint32_t hostpass_after_hit(uint32_t seg, uint32_t kind) { return rz_seg_after_hit(seg, kind); }
extern "C" uint32_t hostpass_hits(uint32_t seg) { return rz_seg_hits(seg); }
extern "C" uint32_t hostpass_first_kind(uint32_t seg) { return rz_seg_first_kind(seg); }
// The pass of a path whose hits have the material kinds kinds[0..n) before it reaches the sky, walked as rz_shade_segment
// walks it: seg starts at 0 (a camera ray), every hit is rz_seg_after_hit, the sky reads rz_pass_of of the word.
extern "C" uint32_t hostpass_walk(const uint32_t *kinds, uint32_t n) {
    uint32_t seg = 0;
    for (uint32_t i = 0; i < n; i++) seg = rz_seg_after_hit(seg, kinds[i]);
    return rz_pass_of(rz_seg_hits(seg), rz_seg_first_kind(seg));
}
