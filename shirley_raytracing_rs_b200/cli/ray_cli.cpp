// ray_cli.cpp — `ray-cli`-compatible front end over the B200 backend.
// Mirrors the reference's CLI (src/argparse.rs:12-170, src/main.rs:36-58) and its render_*
// functions (src/scenes.rs:128-212): same sub-commands, flags, defaults and order of effects
// (scene JSON is written before the scene is finalized, src/scenes.rs:140-146).
//   ray-cli [-v...] render {random|saved|demo|perlin|earth|box-light|cornell} [flags] [scene_input]
//   ray-cli test
// Extra flag (not in the reference): --seed N replaces the OS-seeded thread_rng.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/b200rt_host.h"
#include "../host/raytracer.hpp"

using namespace raytracer;

namespace {
struct Args {
    int verbose = 0;
    std::string sub, scene_input;
    // RenderSettings, src/argparse.rs:107-123
    std::string output = "out.png";
    size_t samples = 100, max_reflect = 50;
    bool single_threaded = false;
    // CameraSettings, :126-146
    scenes::CameraSettings camera;
    // RenderRandom, :70-81
    bool night = false;
    std::string scene_output;
    uint64_t seed = 0x5EED5EEDull;
    std::string checkpoint;     // extra: accumulation-buffer checkpoint (resumed if it exists)
    int gpus = 1;               // extra: render on the first N GPUs of this box (one process, peer access)
    double adaptive = -1.0;     // extra: tile-adaptive sampling to this standard error in 8-bit levels (< 0: off); --samples is the maximum
    uint32_t adaptive_initial = 16;
};

[[noreturn]] void usage(const char* msg) {
    if (msg) fprintf(stderr, "error: %s\n\n", msg);
    fprintf(stderr,
            "USAGE: ray-cli [-v]... render <random|saved|demo|perlin|earth|box-light|cornell> [OPTIONS] [SCENE_INPUT]\n"
            "       ray-cli test\n"
            "OPTIONS:\n"
            "  -o, --output <OUTPUT>            Output file for image [default: out.png]\n"
            "  -s, --samples <SAMPLES>          Number of iterations to sample each pixel [default: 100]\n"
            "  -m, --max-reflect <MAX_REFLECT>  Maximum number of bounces [default: 50]\n"
            "      --single-threaded            Render on a single core (accepted; the GPU backend ignores it)\n"
            "  -w, --width <WIDTH>              Set width of image in pixels [default: 640]\n"
            "      --camera-fov <F>             [default: 20.0]\n"
            "      --camera-focal-length <F>    [default: 1.0]\n"
            "      --camera-aperture <F>        [default: 0.001]\n"
            "      --camera-aspect-ratio <R>    std3x2|std16x9|std16x10|square|target-iphone [default: std3x2]\n"
            "      --night                      (random) Render at night time!\n"
            "      --scene-output <FILE>        (random) Output file for scene_data\n"
            "      --seed <N>                   seed for scene generation and sampling\n"
            "      --gpus <N>                   split the samples over the first N GPUs (NVLink peers) and sum inside the resolve\n"
            "      --checkpoint <FILE>          save the accumulation buffer there; if FILE exists, continue from it:\n"
            "                                   --samples more samples are added (same scene, camera and seed required)\n"
            "      --adaptive <LEVELS>          tile-adaptive sampling: render each 8x4 tile until its estimated standard error\n"
            "                                   is at most LEVELS 8-bit levels; --samples becomes the maximum per pixel\n"
            "      --adaptive-initial <N>       samples of the first adaptive pass [default: 16]\n");
    exit(msg ? 2 : 0);
}

bool parse_ratio(const std::string& v, uint32_t* n, uint32_t* d) {   // CameraAspectRatio::ratio, src/argparse.rs:157-167
    if (v == "std3x2") { *n = 3; *d = 2; }
    else if (v == "std16x9") { *n = 16; *d = 9; }
    else if (v == "std16x10") { *n = 16; *d = 10; }
    else if (v == "square") { *n = 1; *d = 1; }
    else if (v == "target-iphone") { *n = 1170; *d = 2532; }
    else return false;
    return true;
}

Args parse(int argc, char** argv) {
    Args a;
    std::vector<std::string> pos;
    for (int i = 1; i < argc; ++i) {
        std::string s = argv[i];
        auto need = [&](const char* name) -> std::string { if (i + 1 >= argc) usage((std::string(name) + " needs a value").c_str()); return argv[++i]; };
        if (s == "-h" || s == "--help") usage(nullptr);
        else if (s == "--verbose") a.verbose++;
        else if (s.size() >= 2 && s[0] == '-' && s[1] == 'v' && s.find_first_not_of('v', 1) == std::string::npos) a.verbose += (int)s.size() - 1;
        else if (s == "-o" || s == "--output") a.output = need("--output");
        else if (s == "-s" || s == "--samples") a.samples = strtoull(need("--samples").c_str(), nullptr, 10);
        else if (s == "-m" || s == "--max-reflect") a.max_reflect = strtoull(need("--max-reflect").c_str(), nullptr, 10);
        else if (s == "--single-threaded") a.single_threaded = true;
        else if (s == "-w" || s == "--width") a.camera.width = strtoull(need("--width").c_str(), nullptr, 10);
        else if (s == "--camera-fov") a.camera.camera_fov = atof(need("--camera-fov").c_str());
        else if (s == "--camera-focal-length") a.camera.camera_focal_length = atof(need("--camera-focal-length").c_str());
        else if (s == "--camera-aperture") a.camera.camera_aperture = atof(need("--camera-aperture").c_str());
        else if (s == "--camera-aspect-ratio") { if (!parse_ratio(need("--camera-aspect-ratio"), &a.camera.ratio_n, &a.camera.ratio_d)) usage("invalid --camera-aspect-ratio"); }
        else if (s == "--night") a.night = true;
        else if (s == "--scene-output") a.scene_output = need("--scene-output");
        else if (s == "--seed") a.seed = strtoull(need("--seed").c_str(), nullptr, 0);
        else if (s == "--checkpoint") a.checkpoint = need("--checkpoint");
        else if (s == "--gpus") { a.gpus = atoi(need("--gpus").c_str()); if (a.gpus < 1) usage("--gpus needs a positive count"); }
        else if (s == "--adaptive") {
            char* end = nullptr; std::string v = need("--adaptive");
            a.adaptive = strtod(v.c_str(), &end);
            if (v.empty() || *end || !std::isfinite(a.adaptive) || a.adaptive < 0) usage("--adaptive needs a finite number of levels >= 0");
        }
        else if (s == "--adaptive-initial") { int n = atoi(need("--adaptive-initial").c_str()); if (n < 1) usage("--adaptive-initial needs a positive count"); a.adaptive_initial = (uint32_t)n; }
        else if (!s.empty() && s[0] == '-') usage(("unexpected argument " + s).c_str());
        else pos.push_back(s);
    }
    if (a.adaptive >= 0 && a.gpus > 1) usage("--adaptive renders on one GPU: it cannot be combined with --gpus");
    if (a.adaptive >= 0 && !a.checkpoint.empty()) usage("--adaptive cannot be combined with --checkpoint");
    if (pos.empty()) usage("a subcommand is required");
    if (pos[0] == "test") { a.sub = "test"; return a; }
    if (pos[0] != "render" || pos.size() < 2) usage("expected `render <scene>`");
    a.sub = pos[1];
    if (a.sub == "saved") { if (pos.size() < 3) usage("render saved needs SCENE_INPUT"); a.scene_input = pos[2]; }
    return a;
}

// render_scene, src/main.rs:65-130
int render_scene(const Args& args, const scene::SceneBuilder& builder, const camera::Camera& cam, const camera::CameraPosition& pos) {
    size_t samples = args.samples;
    if (samples == 0) { fprintf(stderr, " WARN  samples set to 0, using 1\n"); samples = 1; }   // main.rs:75-80
    std::unique_ptr<scene::Scene> flat = builder.finalize(args.seed ^ 0xA5A5A5A55A5A5A5Aull);
    B200rtCamera c = camera::to_abi(cam, pos);
    if (args.gpus > 1) {                                      // one process, several GPUs: b200rt_render_rgb8_multi
        if (!args.checkpoint.empty()) { fprintf(stderr, " ERROR --checkpoint and --gpus cannot be combined\n"); return B200RT_EINVAL; }
        std::vector<int> devs(args.gpus);
        for (int k = 0; k < args.gpus; ++k) devs[k] = k;
        std::vector<uint8_t> frame((size_t)c.image_width * c.image_height * 3);
        B200rtRenderParams mp{};
        mp.samples = (uint32_t)samples; mp.max_depth = (uint32_t)args.max_reflect; mp.seed = args.seed; mp.device = -1;
        B200rtStats mst{};
        int mrc = b200rt_render_rgb8_multi(&flat->desc, devs.data(), (uint32_t)devs.size(), &c, &mp, frame.data(), &mst);
        if (mrc) { fprintf(stderr, " ERROR %s\n", b200rt_last_error()); return mrc; }
        if (args.verbose >= 1)
            fprintf(stderr, " INFO  %ux%u, %zu spp on %d GPUs: %.1f ms on the slowest device, %.1f Mrays/s (%llu rays)\n", c.image_width, c.image_height, samples, args.gpus,
                    mst.kernel_ms, (double)mst.rays / mst.kernel_ms / 1e3, (unsigned long long)mst.rays);
        mrc = b200rt_write_png(args.output.c_str(), frame.data(), c.image_width, c.image_height);
        if (mrc) { fprintf(stderr, " ERROR cannot write %s\n", args.output.c_str()); return mrc; }
        return 0;
    }
    B200rtScene* dev = nullptr;
    int rc = b200rt_scene_create(&flat->desc, -1, &dev);
    if (rc) { fprintf(stderr, " ERROR %s\n", b200rt_last_error()); return rc; }
    std::vector<uint8_t> rgb((size_t)c.image_width * c.image_height * 3);
    B200rtRenderParams p{};
    p.samples = (uint32_t)samples; p.max_depth = (uint32_t)args.max_reflect; p.seed = args.seed; p.device = -1;
    B200rtStats st{};
    if (args.adaptive >= 0) {
        B200rtAdaptiveParams ad{};
        ad.initial_samples = args.adaptive_initial; ad.max_samples = (uint32_t)samples; ad.threshold = (float)(args.adaptive / 255.0);
        std::vector<float> accum((size_t)c.image_width * c.image_height * 4);
        rc = b200rt_render_adaptive(dev, &c, &p, &ad, accum.data(), rgb.data(), nullptr, &st);
        if (!rc && args.verbose >= 1) {
            float most = 0.f;                          // the last pass brought the most-sampled tiles to this count
            for (size_t k = 3; k < accum.size(); k += 4) most = std::max(most, accum[k]);
            uint32_t passes = 1;
            for (uint64_t n = ad.initial_samples; n < (uint64_t)most; n *= 2) ++passes;
            fprintf(stderr, " INFO  adaptive to %g levels: %.1f spp on average (at most %zu), %u passes\n", args.adaptive,
                    (double)st.paths / ((double)c.image_width * c.image_height), samples, passes);
        }
    } else if (args.checkpoint.empty()) {
        rc = b200rt_render_rgb8(dev, &c, &p, rgb.data(), nullptr, &st);
    } else {
        // progressive: continue the checkpoint's sample sequence (same seed, sample_offset = samples done)
        const size_t n = (size_t)c.image_width * c.image_height * 4;
        std::vector<float> accum(n, 0.0f);
        uint32_t cw = 0, ch = 0, done = 0; uint64_t cseed = 0; float* loaded = nullptr;
        if (std::ifstream(args.checkpoint).good()) {
            rc = b200rt_host_checkpoint_load(args.checkpoint.c_str(), &cw, &ch, &done, &cseed, &loaded);
            if (rc) { b200rt_scene_destroy(dev); fprintf(stderr, " ERROR %s\n", b200rt_host_last_error()); return rc; }
            bool same = cw == c.image_width && ch == c.image_height && cseed == args.seed;
            if (same) memcpy(accum.data(), loaded, n * sizeof(float));
            b200rt_free(loaded);
            if (!same) { b200rt_scene_destroy(dev); fprintf(stderr, " ERROR checkpoint %s was written for another image size or seed\n", args.checkpoint.c_str()); return B200RT_EINVAL; }
            if (args.verbose >= 1) fprintf(stderr, " INFO  resuming %s: %u samples done\n", args.checkpoint.c_str(), done);
        }
        p.sample_offset = done; p.flags |= B200RT_FLAG_ACCUMULATE;
        rc = b200rt_render_rgb8(dev, &c, &p, rgb.data(), accum.data(), &st);
        if (!rc) {
            rc = b200rt_host_checkpoint_save(args.checkpoint.c_str(), accum.data(), c.image_width, c.image_height, done + (uint32_t)samples, args.seed);
            if (rc) fprintf(stderr, " ERROR %s\n", b200rt_host_last_error());
        }
    }
    b200rt_scene_destroy(dev);
    if (rc) { fprintf(stderr, " ERROR %s\n", b200rt_last_error()); return rc; }
    if (args.verbose >= 1)
        fprintf(stderr, " INFO  %ux%u, %zu spp: %.1f ms on the device, %.1f Mrays/s (%llu rays)\n", c.image_width, c.image_height, samples, st.kernel_ms,
                (double)st.rays / st.kernel_ms / 1e3, (unsigned long long)st.rays);
    rc = b200rt_write_png(args.output.c_str(), rgb.data(), c.image_width, c.image_height);   // image::to_image, image.rs:31-44
    if (rc) { fprintf(stderr, " ERROR cannot write %s\n", args.output.c_str()); return rc; }
    return 0;
}
}  // namespace

int main(int argc, char** argv) {
    Args args = parse(argc, argv);
    if (args.sub == "test") { fprintf(stderr, " ERROR there is nothing to test!\n"); return 0; }   // main.rs:60-63
    try {
        scene::SceneBuilder builder;
        camera::Camera cam; camera::CameraPosition pos;
        scenes::HostRng rng(args.seed);
        bool cornell = false;
        if (args.sub == "random") {                                       // render_random, src/scenes.rs:136-165
            builder = scenes::random_scene(rng, args.night);
            if (!args.scene_output.empty()) {
                std::ofstream f(args.scene_output);
                if (!f) throw Error("cannot create " + args.scene_output);
                f << builder.to_json();
            }
        } else if (args.sub == "saved") {                                  // render_saved, :128-134
            std::ifstream f(args.scene_input);
            if (!f) throw Error("cannot open " + args.scene_input);
            std::stringstream ss; ss << f.rdbuf();
            builder = scene::SceneBuilder::from_json(ss.str());
        } else if (args.sub == "demo") builder = scenes::create_scene();
        else if (args.sub == "perlin") builder = scenes::create_perlin_demo();
        else if (args.sub == "earth") builder = scenes::create_earth_demo();
        else if (args.sub == "box-light") builder = scenes::create_box_light();
        else if (args.sub == "cornell") { builder = scenes::create_cornell_box(); cornell = true; }
        else usage(("unknown scene " + args.sub).c_str());
        if (cornell) {                                                     // render_cornell_box, :188-212
            camera::CameraBuilder b;
            b.vfov(40.0).focal_length(1.0).aperture(0.00001).width(args.camera.width).aspect_ratio(camera::AspectRatio::Rational(1, 1));
            cam = b.build();
            pos = camera::CameraPosition::look_at(core::Point({278.0, 278.0, -800.0}), core::Point({278.0, 278.0, 0.0}), core::Vec3(0.0, 1.0, 0.0));
            pos.focus_length = 10.0;
        } else scenes::default_camera(args.camera, &cam, &pos);
        int rc = render_scene(args, builder, cam, pos);
        if (rc) { fprintf(stderr, " ERROR unrecoverable ray-cli failure\n"); return 1; }   // main.rs:54-57
        return 0;
    } catch (const std::exception& e) {
        fprintf(stderr, " ERROR %s\n ERROR unrecoverable ray-cli failure\n", e.what());
        return 1;
    }
}
