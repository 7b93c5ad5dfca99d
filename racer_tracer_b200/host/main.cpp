// racer_render — headless driver over the C++ host: what racer-tracer's main() does between reading the
// configuration and saving the PNG (src/main.rs:64-277), without the minifb window and key handling:
//   config (src/config.rs) -> scene (src/scene/yml.rs) -> camera (src/camera.rs) -> renderer
//   (src/renderer.rs:109-116) -> ScreenBuffer tone map (src/image_buffer.rs:147-153) -> SavePng
//   (src/image_action/png.rs).  Exit code = TracerError ordinal (src/error.rs:71-97), 0 on success.
//
//   racer_render --config config.yml --scene scene.yml [--width W --height H] [--samples N]
//                [--max-depth D] [--seed S] [--preview] [--out image.png] [--image-dir DIR]
//                [--adaptive T [--min-samples N]]   (adaptive sampling up to --samples per pixel: gpu.adaptive)
//                [--dump-flat scene.json]      (flat tables as JSON; needs no GPU)
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>

#include "racer_host.hpp"
#include "yaml_lite.hpp"

using namespace racer;

// --dump-yaml: the parsed tree of one YAML file as JSON (keys lower-cased as the loaders see them, scalars as
// strings); tests compare it with PyYAML on the reference's own files.
static void yaml_to_json(const yaml_lite::Node& n, std::string& out) {
    auto quote = [&](const std::string& s) {
        out += '"';
        for (char c : s) { if (c == '"' || c == '\\') out += '\\'; out += c; }
        out += '"';
    };
    if (n.is_null()) out += "null";
    else if (n.is_scalar()) quote(n.scalar);
    else if (n.is_seq()) {
        out += '[';
        for (size_t i = 0; i < n.seq.size(); ++i) { if (i) out += ','; yaml_to_json(n.seq[i], out); }
        out += ']';
    } else {
        out += '{';
        for (size_t i = 0; i < n.map.size(); ++i) { if (i) out += ','; quote(n.map[i].first); out += ':'; yaml_to_json(n.map[i].second, out); }
        out += '}';
    }
}

int main(int argc, char** argv) {
    std::string config_path, scene_path, out_path, dump_path;
    std::vector<std::string> image_dirs;
    long width = 0, height = 0, samples = -1, max_depth = -1;
    unsigned long long seed = 0;
    bool have_seed = false, preview = false;
    bool have_adaptive = false;
    double adaptive = 0.0;
    long min_samples = -1;
    try {
        for (int i = 1; i < argc; ++i) {
            const std::string a = argv[i];
            auto next = [&]() -> std::string {
                if (i + 1 >= argc) throw TracerError(TracerError::ArgumentParsingError, "Argument parsing Error: " + a + " needs a value");
                return argv[++i];
            };
            if (a == "--config") config_path = next();
            else if (a == "--scene") scene_path = next();
            else if (a == "--out") out_path = next();
            else if (a == "--dump-flat") dump_path = next();
            else if (a == "--dump-yaml") {
                const std::string file = next();
                std::ifstream f(file.c_str());
                if (!f) throw TracerError(TracerError::Configuration, "Config Error (" + file + "): configuration file \"" + file + "\" not found");
                std::string text((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
                try {
                    yaml_lite::Node doc = yaml_lite::parse(text);
                    yaml_lite::lower_keys(doc);
                    std::string out;
                    yaml_to_json(doc, out);
                    std::printf("%s\n", out.c_str());
                } catch (const yaml_lite::ParseError& e) {
                    throw TracerError(TracerError::Configuration, "Config Error (" + file + "): " + e.what());
                }
                return 0;
            }
            else if (a == "--image-dir") image_dirs.push_back(next());
            else if (a == "--width") width = std::atol(next().c_str());
            else if (a == "--height") height = std::atol(next().c_str());
            else if (a == "--samples") samples = std::atol(next().c_str());
            else if (a == "--max-depth") max_depth = std::atol(next().c_str());
            else if (a == "--seed") { seed = std::strtoull(next().c_str(), nullptr, 10); have_seed = true; }
            else if (a == "--preview") preview = true;
            else if (a == "--adaptive") { adaptive = std::atof(next().c_str()); have_adaptive = true; }
            else if (a == "--min-samples") min_samples = std::atol(next().c_str());
            else throw TracerError(TracerError::ArgumentParsingError, "Argument parsing Error: unknown argument " + a);
        }
        Config config = config_path.empty() ? Config() : Config::from_file(config_path);
        if (width > 0) config.screen.width = (size_t)width;
        if (height > 0) config.screen.height = (size_t)height;
        if (samples >= 0) (preview ? config.preview : config.render).samples = (size_t)samples;
        if (max_depth >= 0) (preview ? config.preview : config.render).max_depth = (size_t)max_depth;
        if (have_seed) config.gpu.seed = seed;
        if (have_adaptive) { config.gpu.adaptive = true; config.gpu.adaptive_threshold = adaptive; }
        if (min_samples >= 0) {
            if (!config.gpu.adaptive) throw TracerError(TracerError::ArgumentParsingError, "Argument parsing Error: --min-samples needs --adaptive");
            config.gpu.adaptive_min_samples = (int32_t)min_samples;
        }
        if (scene_path.empty() && config.loader.kind == SceneLoaderConfig::Yml) scene_path = config.loader.path;
        if (scene_path.empty() && config.loader.kind == SceneLoaderConfig::Random) scene_path = "random";
        if (scene_path.empty() && config.loader.kind == SceneLoaderConfig::Sandbox) scene_path = "sandbox:../resources/scenes/cornell_box.yml";   // sandbox.rs:41-42
        if (scene_path.empty()) throw TracerError(TracerError::ArgumentParsingError, "Argument parsing Error: --scene (or loader: Yml) is required");
        if (config.screen.width < 2 || config.screen.height < 2)
            throw TracerError(TracerError::Configuration, "Config Error (screen): width and height must be >= 2");

        // SceneLoaderConfig::{Random, Sandbox, Yml} (config.rs:84-93); "sandbox:<path of cornell_box.yml>"
        std::unique_ptr<SceneData> scene = scene_path == "random" ? SceneData::load_random(config.gpu.seed)
                                           : scene_path.rfind("sandbox:", 0) == 0 ? SceneData::load_sandbox(scene_path.substr(8), config.gpu.seed)
                                                                                  : SceneData::load_yml(scene_path, config.gpu.seed, image_dirs);
        const Image image(config.screen.width, config.screen.height);
        const rc_camera camera = make_camera(merge_camera(scene->camera, config.camera), image);   // main.rs:95-111
        const rc_tone_map tone_map = scene->has_tone_map ? scene->tone_map : config.tone_map;       // main.rs:84-86

        if (!dump_path.empty()) {
            std::ofstream f(dump_path.c_str());
            f << "{\"scene\":" << scene->to_json() << ",\"camera\":[";
            const double* cd = reinterpret_cast<const double*>(&camera);
            char buf[40];
            for (size_t k = 0; k < sizeof(rc_camera) / sizeof(double); ++k) { std::snprintf(buf, sizeof(buf), "%.17g", cd[k]); f << (k ? "," : "") << buf; }
            f << "],\"tone_map_type\":" << tone_map.type << ",\"width\":" << image.width << ",\"height\":" << image.height
              << ",\"render\":[" << config.render.samples << "," << config.render.max_depth << "],\"preview\":[" << config.preview.samples << ","
              << config.preview.max_depth << "," << config.preview.scale << "]}";
            if (out_path.empty()) return 0;
        }

        // renderer selection, renderer.rs:109-116; this binary only has the CUDA renderers
        const RendererConfig which = preview ? RendererConfig::CudaPreview : RendererConfig::Cuda;
        std::unique_ptr<Renderer> renderer = make_renderer(which, preview ? config.preview : config.render, config.gpu, image);
        CudaRenderer& gpu = static_cast<CudaRenderer&>(*renderer);
        ScreenBuffer screen(image, tone_map);
        DataWriter<ImageBufferEvent> writer([&](ImageBufferEvent&& ev) { screen.update(ev, gpu); });
        RenderData rd;
        rd.camera_data = &camera; rd.image = &image; rd.scene = scene.get(); rd.config = &config;
        const auto t0 = std::chrono::steady_clock::now();
        renderer->render(rd, writer);
        const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        const rc_stats st = gpu.stats();
        std::printf("It took %.3f seconds to render the image. (%llu samples, %.3f ms on the GPU, %llu kernel launches)\n", secs,
                    (unsigned long long)st.samples, st.gpu_ms, (unsigned long long)st.kernel_launches);   // interactive.rs:255-259
        if (!out_path.empty() || config.image_action == ImageActionConfig::SavePng) {
            const std::string dir = config.has_image_output_dir ? config.image_output_dir : std::string(".");
            const std::string path = save_png(screen.rgba(), image.width, image.height, dir, out_path);
            std::printf("Saved image to: %s\n", path.c_str());
        }
        return 0;
    } catch (const TracerError& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return exit_code(e);
    }
}
