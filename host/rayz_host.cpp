// rayz_host — stand-in for the reference executable (src/rayz.zig:12-43):
//
//     rayz_host <img_w> [out.ppm] [--spp N] [--depth N] [--seed S] [--render-seed S]
//               [--variant auto|mega|wavefront|bvh] [--gpus N] [--grid G] [--scene bouncing|penultimate]
//               [--dump-scene file] [--dump-linear file] [--ppm-bench] [--noise-target X [--max-spp N] [--adaptive]]
//               [--guides PREFIX] [--denoise FILE] [--sobol] [--rqmc] [--pooled] [--passes PREFIX] [--mattes PREFIX]
//               [--filter box|tent|gaussian|blackman-harris[:WIDTH]]
//
// Same argv contract (img_w required, optional output path, else stdout), same report line
// ("Finished render (…s): … rps and … us per ray", rays = primary samples), same ASCII P3 output.
// The pixel loop runs in librayz_cuda.so; the timed region covers what the reference's covers
// (hittables + BVH build == scene upload, and the render).  --noise-target X (displayed-value rms error, 1/255 = one 8-bit
// step) starts at --spp samples and doubles them until the frame reaches X or --max-spp (default 4096); the samples reached
// and the error go to stderr, the report line and the P3 output are unchanged.  With --adaptive, X bounds every pixel's error
// and only the pixels still above it get more samples (RZ_RENDER_ADAPTIVE); stderr then also reports the paths traced and the
// mean and max samples per pixel.  --guides PREFIX also writes the guide buffers of the render's camera samples for a denoiser
// (rayz_cuda_render_guides) as PFM files: PREFIX_albedo.pfm and PREFIX_normal.pfm (3 channels), PREFIX_depth.pfm (1 channel).
// --denoise FILE renders with RZ_RENDER_MOMENTS (no pixel changes), computes guides over the render's own samples and writes the
// frame denoised by rayz_cuda_denoise (default parameters) to FILE as P3; the normal output and the report line are unchanged.
// --sobol draws the camera and scatter samples from Owen-scrambled Sobol pairs (RZ_RENDER_SOBOL) in every one of these runs,
// guides included.  --rqmc does the same with two independently scrambled replicates per pixel and the noise estimate they
// allow (RZ_RENDER_SOBOL | RZ_RENDER_RQMC | RZ_RENDER_MOMENTS): --noise-target then stops on it; --spp and --max-spp must be even.
// --pooled (with --noise-target X --adaptive) stops each pixel on an error pooled over its row segment (RZ_RENDER_ADAPTIVE_POOLED),
// so that X bounds the measured error too; without --adaptive the library refuses it.
// --passes PREFIX renders with RZ_RENDER_PASSES (no pixel changes) and writes the frame's seven light-path passes
// (rayz_cuda_passes) as 3-channel PFM files PREFIX_<name>.pfm, name = environment, diffuse_direct, diffuse_indirect,
// glossy_direct, glossy_indirect, transmission_direct, transmission_indirect; they sum to the frame's linear values.
// --mattes PREFIX also writes the ID mattes of the render's camera samples (rayz_cuda_render_mattes), six ranks, as 3-channel
// PFM files PREFIX_rank<r>.pfm: the rank's sphere index as a float (-1 the sky, -2 no such rank), its coverage, 0.  Mattes
// take at most 1024 samples per pixel.
// --filter KIND[:WIDTH] draws each camera sample's offset from a reconstruction filter (RZ_RENDER_FILTER) in every one of these
// runs, guides and mattes included: tent, gaussian or blackman-harris, WIDTH its full width in px (1 to 4, a multiple of
// 1/16; default 2, 3 and 1.5).  The default, box, is the reference's uniform jitter.
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
    const char *dump_scene = nullptr, *dump_linear = nullptr, *guides = nullptr, *denoise = nullptr, *passes = nullptr,
               *mattes = nullptr;
    bool ppm_bench = false, penultimate = false, adaptive = false, sobol = false, rqmc = false, pooled = false;
    uint32_t pixel_filter = 0;
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
        else if (a == "--adaptive") adaptive = true;
        else if (a == "--sobol") sobol = true;
        else if (a == "--rqmc") rqmc = true;
        else if (a == "--pooled") pooled = true;
        else if (a == "--guides") guides = val();
        else if (a == "--denoise") denoise = val();
        else if (a == "--passes") passes = val();
        else if (a == "--mattes") mattes = val();
        else if (a == "--filter") {
            const std::string v = val(), kind = v.substr(0, v.find(':'));
            const uint32_t k = kind == "box" ? RZ_FILTER_BOX : kind == "tent" ? RZ_FILTER_TENT : kind == "gaussian" ? RZ_FILTER_GAUSSIAN
                               : kind == "blackman-harris" ? RZ_FILTER_BLACKMAN_HARRIS : 99u;
            double width = 0;
            if (v.find(':') != std::string::npos) width = std::strtod(v.c_str() + v.find(':') + 1, nullptr);
            const double w16 = width * 16.0;
            if (k == 99u || !(w16 >= 0 && w16 <= 255 && w16 == std::floor(w16))) {
                std::fprintf(stderr, "--filter: expected box, tent, gaussian or blackman-harris, optionally :WIDTH in px (a multiple of 1/16), got %s\n", v.c_str());
                return 2;
            }
            pixel_filter = RZ_RENDER_FILTER(k, (uint32_t)w16);   // the library refuses widths outside 1..4 px, and a width with the box
        }
        else if (a == "--scene") penultimate = std::string(val()) == "penultimate";
        else if (a == "--variant") {
            const std::string v = val();
            variant = v == "mega" ? RZ_VARIANT_MEGA : v == "mega_single" ? RZ_VARIANT_MEGA_SINGLE : v == "wavefront" ? RZ_VARIANT_WAVEFRONT : v == "bvh" ? RZ_VARIANT_BVH : RZ_VARIANT_AUTO;
        } else if (!out_fname && a.rfind("--", 0) != 0) out_fname = argv[i];
        else { std::fprintf(stderr, "unknown argument %s\n", a.c_str()); return 2; }
    }
    if (mattes && spp > RZ_MATTE_MAX_SPP) { std::fprintf(stderr, "--mattes: --spp %zu is above the mattes' %u samples per pixel\n", spp, RZ_MATTE_MAX_SPP); return 2; }
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
        tracer.adaptive = adaptive;
        tracer.moments = denoise != nullptr;
        tracer.sobol = sobol;
        tracer.rqmc = rqmc;
        tracer.pooled = pooled;
        tracer.passes = passes != nullptr;
        tracer.pixel_filter = pixel_filter;
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
        if (noise_target > 0 && adaptive)
            std::fprintf(stderr, "  [rayz_cuda] adaptive: %.0f paths, mean %.2f spp, max %llu spp, max error %.5f (%.2f 8-bit steps)\n", rays_traced,
                         rays_traced / std::max<double>(1.0, tracer.noise.n_pixels), (unsigned long long)tracer.noise.samples, tracer.noise.max_err,
                         tracer.noise.max_err * 255.0);
        if (passes) {
            tracer.readPasses();
            static const char *const names[RZ_PASS_COUNT] = {"environment", "diffuse_direct", "diffuse_indirect", "glossy_direct",
                                                             "glossy_indirect", "transmission_direct", "transmission_indirect"};
            const size_t plane = tracer.img.w * tracer.img.h * 4;
            for (int i = 0; i < RZ_PASS_COUNT; i++) {
                const std::string path = std::string(passes) + "_" + names[i] + ".pfm";
                FILE *f = std::fopen(path.c_str(), "wb");
                if (!f) { std::perror(path.c_str()); return 1; }
                writePFM(f, tracer.pass_planes.data() + i * plane, tracer.img.w, tracer.img.h, 4, 0, 3);
                std::fclose(f);
            }
        }
        if (guides || denoise) tracer.renderGuides();
        if (guides) {
            const struct { const char *name; const std::vector<float> &src; size_t first, channels; } files[3] = {
                {"_albedo.pfm", tracer.albedo, 0, 3}, {"_normal.pfm", tracer.normal, 0, 3}, {"_depth.pfm", tracer.normal, 3, 1}};
            for (const auto &o : files) {
                const std::string path = std::string(guides) + o.name;
                FILE *f = std::fopen(path.c_str(), "wb");
                if (!f) { std::perror(path.c_str()); return 1; }
                writePFM(f, o.src.data(), tracer.img.w, tracer.img.h, 4, o.first, o.channels);
                std::fclose(f);
            }
        }
        if (denoise) {
            tracer.denoise();
            FILE *f = std::fopen(denoise, "wb");
            if (!f) { std::perror(denoise); return 1; }
            tracer.denoised.writePPM(f);
            std::fclose(f);
        }
        if (mattes) {
            const uint32_t ranks = 6;
            tracer.renderMattes(ranks);
            const size_t npx = tracer.img.w * tracer.img.h;
            std::vector<float> plane(npx * 3, 0.f);
            for (uint32_t r = 0; r < ranks; r++) {
                for (size_t i = 0; i < npx; i++) {
                    plane[3 * i] = (float)tracer.matte_ids[i * ranks + r];
                    plane[3 * i + 1] = tracer.matte_coverage[i * ranks + r];
                }
                const std::string path = std::string(mattes) + "_rank" + std::to_string(r) + ".pfm";
                FILE *f = std::fopen(path.c_str(), "wb");
                if (!f) { std::perror(path.c_str()); return 1; }
                writePFM(f, plane.data(), tracer.img.w, tracer.img.h, 3, 0, 3);
                std::fclose(f);
            }
        }
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
