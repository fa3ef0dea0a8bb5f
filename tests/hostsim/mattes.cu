// Test-only: the rank key of the ID mattes (rz_device.cuh's rz_matte_key and its decode) compiled as HOST code, so that
// tests/test_mattes_cpu.py can check its order against numpy.  The product only ever runs these functions inside its CUDA
// kernels.
#include <cstdint>

#include "../../rayz_b200/csrc/rz_device.cuh"

extern "C" int32_t hostmatte_miss(void) { return RZ_MATTE_MISS; }
extern "C" int32_t hostmatte_empty(void) { return RZ_MATTE_EMPTY; }
extern "C" uint32_t hostmatte_max_ranks(void) { return RZ_MATTE_MAX_RANKS; }
extern "C" uint32_t hostmatte_max_spp(void) { return RZ_MATTE_MAX_SPP; }
// keys[i] = rz_matte_key(count[i], id[i])
extern "C" void hostmatte_keys(const uint32_t *count, const int32_t *id, uint32_t n, unsigned long long *keys) {
    for (uint32_t i = 0; i < n; i++) keys[i] = rz_matte_key(count[i], id[i]);
}
extern "C" void hostmatte_decode(const unsigned long long *keys, uint32_t n, uint32_t *count, int32_t *id) {
    for (uint32_t i = 0; i < n; i++) { count[i] = rz_matte_key_count(keys[i]); id[i] = rz_matte_key_id(keys[i]); }
}
