// rayz_host — stand-in for the reference executable (src/rayz.zig:12-43):
//
//     rayz_host <img_w> [out.ppm] [--spp N] [--depth N] [--seed S] [--render-seed S]
//               [--variant auto|mega|wavefront|bvh] [--gpus N] [--grid G] [--scene bouncing|penultimate]
//               [--dump-scene file] [--dump-linear file] [--ppm-bench] [--noise-target X [--max-spp N]]
//
// Same argv contract (img_w required, optional output path, else stdout), same report line
// ("Finished render (…s): … rps and … us per ray", rays = primary samples), same ASCII P3 output.
// The pixel loop runs in librayz_cuda.so; the timed region covers what the reference's covers
// (hittables + BVH build == scene upload, and the render).  --noise-target X (displayed-value rms error, 1/255 = one 8-bit
// step) starts at --spp samples and doubles them until the frame reaches X or --max-spp (default 4096); the samples reached
// and the error go to stderr, the report line and the P3 output are unchanged.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <random>
#include <string>

#include "rayz_host.hpp"

using namespace rayz;

int main(int argc, char **argv) {
    if (argc < 2) {
        std::fprintf(stderr, "usage: %s <img_w> [out.ppm] [--spp N] [--depth N] [--seed S] [--variant V] [--gpus N]\n", argv[0]);
        return 2;  // the reference panics on a missing argv[1] (`args.next().?`, rayz.zig:16)
    }
    char *end = nullptr;
    const unsigned long long img_w = std::strtoull(argv[1], &end, 10);
    if (!end || *end || img_w == 0) { std::fprintf(stderr, "error: InvalidCharacter\n"); return 1; }
    const char *out_fname = nullptr;
    uint64_t seed = 0, render_seed = 1;
    bool have_seed = false;
    size_t spp = 10, depth = 50;
    int gpus = 1, grid = 11;
    uint32_t variant = RZ_VARIANT_AUTO;
    const char *dump_scene = nullptr, *dump_linear = nullptr;
    bool ppm_bench = false, penultimate = false;
    float noise_target = 0;
    uint32_t max_spp = 4096;
    for (int i = 2; i < argc; i++) {
        const std::string a = argv[i];
        auto val = [&]() -> const char * { if (i + 1 >= argc) { std::fprintf(stderr, "missing value for %s\n", a.c_str()); std::exit(2); } return argv[++i]; };
        if (a == "--spp") spp = std::strtoull(val(), nullptr, 10);
        else if (a == "--depth") depth = std::strtoull(val(), nullptr, 10);
        else if (a == "--seed") { seed = std::strtoull(val(), nullptr, 10); have_seed = true; }
        else if (a == "--render-seed") render_seed = std::strtoull(val(), nullptr, 10);
        else if (a == "--gpus") gpus = std::atoi(val());
        else if (a == "--grid") grid = std::atoi(val());
        else if (a == "--dump-scene") dump_scene = val();
        else if (a == "--dump-linear") dump_linear = val();
        else if (a == "--ppm-bench") ppm_bench = true;
        else if (a == "--noise-target") noise_target = std::strtof(val(), nullptr);
        else if (a == "--max-spp") max_spp = (uint32_t)std::strtoul(val(), nullptr, 10);
        else if (a == "--scene") penultimate = std::string(val()) == "penultimate";
        else if (a == "--variant") {
            const std::string v = val();
            variant = v == "mega" ? RZ_VARIANT_MEGA : v == "mega_single" ? RZ_VARIANT_MEGA_SINGLE : v == "wavefront" ? RZ_VARIANT_WAVEFRONT : v == "bvh" ? RZ_VARIANT_BVH : RZ_VARIANT_AUTO;
        } else if (!out_fname && a.rfind("--", 0) != 0) out_fname = argv[i];
        else { std::fprintf(stderr, "unknown argument %s\n", a.c_str()); return 2; }
    }
    if (!have_seed) { std::random_device rd; seed = ((uint64_t)rd() << 32) ^ rd(); }  // renderer.zig:55-59: seeded from the OS

    try {
        const bool pen = penultimate;   // rayz.zig:46-55 (randomBouncing) or :171-180 (penultimateScene)
        Tracer tracer((size_t)img_w, 20.0, pen ? 3.4 : 10.0, pen ? 10.0 : 0.6, pen ? V3{-2, 2, 1} : V3{13, 2, 3}, pen ? V3{0, 0, -1} : V3{}, V3::y_hat(), seed);
        tracer.samples_per_px = spp;
        tracer.max_bounces = depth;
        tracer.render_seed = render_seed;
        tracer.variant = variant;
        tracer.noise_target = noise_target;
        tracer.max_spp = max_spp;
        tracer.devices.clear();
        for (int g = 0; g < gpus; g++) tracer.devices.push_back(g);
        if (pen) penultimateScene(tracer); else randomBouncing(tracer, -grid, grid);
        tracer.initBackend();  // like Tracer.init's allocations: before the timer (rayz.zig:22-24)

        const auto st = std::chrono::steady_clock::now();
        const double rays_traced = (double)tracer.render();
        const double durr = std::chrono::duration<double>(std::chrono::steady_clock::now() - st).count();
        std::fprintf(stderr, "Finished render (%.2fs): %.2f rps and %.2f us per ray\n", durr, rays_traced / durr, 1e6 * durr / rays_traced);
        std::fprintf(stderr, "  [rayz_cuda] path kernel %.3f ms, resolve %.3f ms, %u launches, %u static + %u moving spheres, variant %u, %d GPU(s)\n",
                     tracer.timing.kernel_ms, tracer.timing.resolve_ms, tracer.timing.launches, tracer.timing.n_static, tracer.timing.n_moving,
                     tracer.timing.variant, gpus);
        if (noise_target > 0)
            std::fprintf(stderr, "  [rayz_cuda] noise target %.5f: %llu spp reached, rms error %.5f (%.2f 8-bit steps), mean %.5f, max %.5f, %u of %u pixels above\n",
                         noise_target, (unsigned long long)tracer.noise.samples, tracer.noise.rms_err, tracer.noise.rms_err * 255.0, tracer.noise.mean_err,
                         tracer.noise.max_err, tracer.noise.n_above, tracer.noise.n_pixels);
        if (dump_scene && !dumpScene(tracer, dump_scene)) { std::perror(dump_scene); return 1; }
        if (dump_linear) {
            FILE *f = std::fopen(dump_linear, "wb");
            if (!f) { std::perror(dump_linear); return 1; }
            std::fwrite(tracer.lin.data(), sizeof(float), tracer.lin.size(), f);
            std::fclose(f);
        }
        const auto tw = std::chrono::steady_clock::now();
        size_t ppm_bytes = 0;
        if (out_fname) {
            FILE *f = std::fopen(out_fname, "wb");
            if (!f) { std::perror(out_fname); return 1; }
            ppm_bytes = tracer.img.writePPM(f);
            std::fclose(f);
        } else {
            ppm_bytes = tracer.img.writePPM(stdout);
        }
        const double wms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tw).count();
        std::fprintf(stderr, "  [rayz_host] writePPM: %zu bytes of P3 text in %.1f ms (%.0f MB/s)\n", ppm_bytes, wms, ppm_bytes / (wms * 1e-3) / 1e6);
        if (ppm_bench) {   // the formatter alone, without the file system: best of 5
            std::vector<char> buf;
            double best = 1e30;
            for (int i = 0; i < 5; i++) {
                const auto t0 = std::chrono::steady_clock::now();
                ppm_bytes = tracer.img.formatPPM(buf);
                best = std::min(best, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
            }
            std::fprintf(stderr, "  [rayz_host] formatPPM: %zux%zu, %zu bytes in %.2f ms (best of 5)\n", tracer.img.w, tracer.img.h, ppm_bytes, best);
        }
    } catch (const CudaBackendError &e) {
        std::fprintf(stderr, "error: CudaBackend (%d): %s\n", e.code, e.what());
        return 1;
    }
    return 0;
}
