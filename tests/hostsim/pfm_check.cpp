// Test-only driver of the C++ host's PFM writer (host/rayz_host.hpp: writePFM, the --guides output).
//   pfm_check <w> <h> <seed> <prefix>     fills a w x h x 4 float buffer with a seeded pattern, writes <prefix>_rgb.pfm (floats
//                                         0..2 of every pixel) and <prefix>_w.pfm (float 3), prints the two byte counts
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../host/rayz_host.hpp"

int main(int argc, char **argv) {
    if (argc < 5) return 2;
    const size_t w = std::strtoull(argv[1], nullptr, 10), h = std::strtoull(argv[2], nullptr, 10);
    uint64_t s = std::strtoull(argv[3], nullptr, 10);
    std::vector<float> px(w * h * 4);
    for (float &v : px) {   // the same LCG the Python test runs; every value is exact in f32 (24 significant bits)
        s = s * 6364136223846793005ull + 1442695040888963407ull;
        v = (float)((int64_t)(s >> 40) - (1 << 23)) / (float)(1 << 20);
    }
    const std::string prefix = argv[4];
    size_t n[2];
    for (int k = 0; k < 2; k++) {
        const std::string path = prefix + (k == 0 ? "_rgb.pfm" : "_w.pfm");
        FILE *f = std::fopen(path.c_str(), "wb");
        if (!f) return 1;
        n[k] = rayz::writePFM(f, px.data(), w, h, 4, k == 0 ? 0 : 3, k == 0 ? 3 : 1);
        std::fclose(f);
    }
    std::printf("%zu %zu\n", n[0], n[1]);
    return 0;
}
