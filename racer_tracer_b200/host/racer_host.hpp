// racer_host.hpp — C++ mirror of the part of the reference's Rust host that sits above the C ABI
// (include/racer_cuda.h).  The reference is Rust and this image has no Rust toolchain, so the host
// side of the boundary is written here in C++ with the reference's names, argument meaning and
// error behaviour; INTEGRATION.md holds the Rust shim a maintainer adds to the real crate.
//
//   reference (racer-tracer/src/)                     here
//   error.rs:4-97        TracerError + exit codes      racer::TracerError, exit_code()
//   config.rs:69-225     Config, RenderConfig, ...     racer::Config::from_file
//   camera.rs:393-464    CameraData::merge             racer::merge_camera
//   camera.rs:196-234    Camera::new                   racer::make_camera
//   scene/yml.rs:43-458  YmlLoader                     racer::SceneData::load_yml
//   bvh_node.rs:31-82    Node::build                   racer::SceneData (host-built BVH)
//   renderer.rs:92-116   RenderData, Renderer, factory racer::RenderData, Renderer, make_renderer
//   image_buffer.rs:63-71 ImageBufferEvent             racer::ImageBufferEvent
//   data_bus.rs          DataWriter<T>                 racer::DataWriter<T>
//   renderer/cpu.rs      CpuRenderer                   racer::CudaRenderer        (RendererConfig::Cuda)
//   renderer/cpu_scaled.rs CpuRendererScaled           racer::CudaPreviewRenderer (RendererConfig::CudaPreview)
//   image_buffer.rs:135-170 ScreenBuffer::update       racer::ScreenBuffer
//   image_action/png.rs  SavePng                       racer::save_png
#pragma once
#include <cstdint>
#include <functional>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/racer_cuda.h"

namespace racer {

// ---- error.rs -------------------------------------------------------------------------------
struct TracerError : std::runtime_error {
    enum Kind {
        FailedToCreateWindow = 1, FailedToUpdateWindow = 2, Configuration = 3, UnknownMaterial = 4,
        FailedToAcquireLock = 5, ExitEvent = 6, CancelEvent = 7, ImageSave = 8, SceneLoad = 9,
        ArgumentParsingError = 10, KeyError = 11, CreateLogError = 12, RecieveError = 13, SendError = 14,
        ActionProtocolError = 15, BusWriteError = 16, BusReadError = 17, BusUpdateError = 18,
        BusTimeoutError = 19, NoObjectWithId = 20, FailedToOpenImage = 21, FailedToParse = 22,
        Cuda = 23   // new: any failure of the C ABI (no CPU fallback; SURVEY §8(b))
    } kind;
    TracerError(Kind k, const std::string& text) : std::runtime_error(text), kind(k) {}
};
inline int exit_code(const TracerError& e) { return (int)e.kind; }   // impl From<TracerError> for i32, error.rs:71-97

// ---- vec3.rs --------------------------------------------------------------------------------
struct Vec3 {
    double x = 0, y = 0, z = 0;
};
typedef Vec3 Color;

// ---- config.rs ------------------------------------------------------------------------------
struct RenderConfig {   // config.rs:75-82
    size_t samples = 0, max_depth = 0, num_threads_width = 0, num_threads_height = 0, scale = 0;
};
struct ScreenConfig {   // config.rs:69-73
    size_t height = 0, width = 0;
};
enum class RendererConfig { Cpu, CpuPreview, Cuda, CudaPreview };   // config.rs:108-113 + the two new variants
enum class ImageActionConfig { None, SavePng };                     // config.rs:95-100
struct SceneLoaderConfig {                                          // config.rs:84-93
    enum Kind { None, Yml, Random, Sandbox } kind = None;
    std::string path;
};
struct CameraConfig {   // config.rs:172-181 (Option<..> fields)
    bool has_vfov = false, has_aperture = false, has_focus_distance = false, has_pos = false, has_look_at = false;
    double vfov = 0, aperture = 0, focus_distance = 0;
    Vec3 pos, look_at;
};
struct GpuConfig {      // new optional `gpu:` block
    uint64_t seed = 0;
    int variant = RC_VARIANT_MEGAKERNEL, sampler = RC_SAMPLER_DIRECT, split = RC_SPLIT_TILES, specialize = 2;
    std::vector<int32_t> devices;
    // optional `adaptive: {threshold, min_samples}`: the full renderer samples adaptively (rc_render_adaptive) with
    // render.samples as the per-pixel maximum
    bool adaptive = false;
    double adaptive_threshold = 0.0;
    int32_t adaptive_min_samples = 16;
    // optional `denoise: {levels, sigma_l, sigma_n, sigma_z}`: the full renderer filters its render (rc_render_denoised);
    // excludes `adaptive`
    bool denoise = false;
    int32_t denoise_levels = 5;
    double denoise_sigma_l = 4.0, denoise_sigma_n = 128.0, denoise_sigma_z = 1.0;
};
struct Config {         // config.rs:183-215
    RenderConfig preview, render;
    ScreenConfig screen;
    SceneLoaderConfig loader;
    ImageActionConfig image_action = ImageActionConfig::None;
    bool has_image_output_dir = false;
    std::string image_output_dir;
    RendererConfig renderer = RendererConfig::Cpu;
    RendererConfig preview_renderer = RendererConfig::CpuPreview;
    CameraConfig camera;
    rc_tone_map tone_map;   // From<&ToneMapConfig> already applied (tone_map.rs:18-66); default None
    GpuConfig gpu;
    Config();
    static Config from_file(const std::string& file);   // config.rs:217-224; throws Configuration
};

// ---- image.rs -------------------------------------------------------------------------------
struct Image {          // image.rs:5-16
    size_t width = 0, height = 0;
    double aspect_ratio = 1.0;
    Image() {}
    Image(size_t w, size_t h) : width(w), height(h), aspect_ratio((double)w / (double)h) {}
};

// ---- camera.rs ------------------------------------------------------------------------------
struct CameraData {     // CameraData::merge result, camera.rs:393-464
    double vfov = 20.0, aperture = 0.0, focus_distance = 1000.0;
    Vec3 pos{0, 0, 0}, look_at{0, 0, -1};
};
CameraData merge_camera(const CameraConfig& scene, const CameraConfig& config);
// Camera::new (camera.rs:196-234) with scene_up = +y and time 0..1 (main.rs:97-110): the CameraSharedData
rc_camera make_camera(const CameraData& cam, const Image& image);

// ---- scene: YAML -> flat SoA + host BVH -------------------------------------------------------
struct SceneData {
    // owned arrays the rc_scene points into
    std::vector<int32_t> prim_type, prim_material, prim_instance;
    std::vector<double> prim_data, prim_aabb, prim_motion;
    bool has_motion = false;
    std::vector<uint32_t> prim_id;
    std::vector<rc_instance> instances;
    std::vector<rc_material> materials;
    std::vector<rc_texture> textures;
    std::vector<rc_perlin> perlin;
    std::vector<rc_bvh_node> nodes;
    std::vector<std::vector<uint8_t>> image_pixels;
    std::vector<rc_image> images;
    std::vector<std::string> object_keys;   // canonical object n (1-based) -> lower-cased YAML key
    rc_scene scene;                          // valid as long as this object lives and is not moved
    CameraConfig camera;                     // the scene's `camera:` block (yml.rs:455)
    bool has_tone_map = false;
    rc_tone_map tone_map;                    // the scene's `tone_map:` block (yml.rs:456)
    bool changed = true;                     // BoundingVolumeHirearchy::changed(), bvh_node.rs:176-205

    SceneData();
    SceneData(const SceneData&) = delete;
    SceneData& operator=(const SceneData&) = delete;
    // YmlLoader::load (yml.rs:43-47,173-458): throws Configuration / SceneLoad / UnknownMaterial /
    // FailedToOpenImage exactly where the reference returns them.
    static std::unique_ptr<SceneData> load_yml(const std::string& path, uint64_t seed = 0,
                                               const std::vector<std::string>& image_dirs = {}, bool sandbox = false);
    // Sandbox::load (scene/sandbox.rs:39-81), the loader racer-tracer/config.yml selects: cornell_box.yml (the
    // reference reads ../resources/scenes/cornell_box.yml) plus two rotated, translated boxes.
    static std::unique_ptr<SceneData> load_sandbox(const std::string& cornell_box_yml, uint64_t seed = 0);
    // Random::load (scene/random.rs:25-95): checkered ground, 22 x 22 small spheres (diffuse ones move), three
    // large spheres; its own camera (vfov 20, aperture 0.1, focus 10).  Deterministic in `seed`.
    static std::unique_ptr<SceneData> load_random(uint64_t seed = 0);
    void wire();                   // point `scene` at the owned arrays
    std::string to_json() const;   // flat tables as JSON (tests compare them with the Python harness)
};

rc_tone_map make_tone_map_default();   // ToneMapConfig::None with the reference's defaults in the other fields

// ---- data_bus.rs / image_buffer.rs ------------------------------------------------------------
struct ImageBufferEvent {   // ImageBufferEvent::BufferUpdate, image_buffer.rs:63-71
    std::vector<Color> rgb;
    size_t r = 0, c = 0, width = 0, height = 0;
};

template <typename T>
class DataWriter {          // data_bus.rs: write() hands the message to the bus's readers
public:
    typedef std::function<void(T&&)> Sink;
    explicit DataWriter(Sink sink) : sink_(std::move(sink)) {}
    void write(T&& message) const {
        std::lock_guard<std::mutex> lock(mutex_);
        sink_(std::move(message));
    }
private:
    Sink sink_;
    mutable std::mutex mutex_;
};

// ScreenBuffer (image_buffer.rs:113-170): keeps the tone-mapped image; update() applies the tone map to
// a BufferUpdate and stores it at (r, c).  The tone map + `f64 as u32` packer run on the GPU
// (rc_postprocess) when a CUDA renderer is given, which is the only implementation here.
class CudaRenderer;
class ScreenBuffer {
public:
    ScreenBuffer(const Image& image, const rc_tone_map& tm) : image_(image), tone_map_(tm), rgb_(image.width * image.height) {}
    void update(const ImageBufferEvent& ev, CudaRenderer& gpu);
    const std::vector<Color>& rgb() const { return rgb_; }          // tone-mapped colours
    const std::vector<uint8_t>& rgba() const { return rgba_; }      // the SavePng byte stream, png.rs:21-31
private:
    Image image_;
    rc_tone_map tone_map_;
    std::vector<Color> rgb_;
    std::vector<uint8_t> rgba_;
};

// ---- renderer.rs ------------------------------------------------------------------------------
struct RenderData {         // renderer.rs:92-99
    const rc_camera* camera_data = nullptr;
    const Image* image = nullptr;
    SceneData* scene = nullptr;          // scene: &dyn Hittable + background: &dyn BackgroundColor, flattened
    const Config* config = nullptr;
    const volatile int32_t* cancel_event = nullptr;   // Option<&SignalEvent>
};

class Renderer {            // trait Renderer, renderer.rs:101-107
public:
    virtual ~Renderer() {}
    // Result<(), TracerError>: throws TracerError; CancelEvent when the flag is set on entry
    // (cpu.rs:79-83); a render cancelled midway returns without writing (cpu.rs:55-62).
    virtual void render(const RenderData& render_data, const DataWriter<ImageBufferEvent>& writer) = 0;
};

class CudaRenderer : public Renderer {        // replaces CpuRenderer (renderer/cpu.rs)
public:
    CudaRenderer(const RenderConfig& config, const GpuConfig& gpu);
    ~CudaRenderer() override;
    void render(const RenderData& render_data, const DataWriter<ImageBufferEvent>& writer) override;
    rc_ctx* context() const { return ctx_; }
    rc_stats stats() const;
protected:
    void sync_scene(const RenderData& rd);
    rc_params params(const RenderData& rd) const;
    RenderConfig config_;
    GpuConfig gpu_;
    std::shared_ptr<rc_ctx> shared_;   // one context per process and device list, shared with the other renderer
    rc_ctx* ctx_ = nullptr;
};

class CudaPreviewRenderer : public CudaRenderer {   // replaces CpuRendererScaled (renderer/cpu_scaled.rs)
public:
    CudaPreviewRenderer(const RenderConfig& config, const GpuConfig& gpu, const Image& image);
    void render(const RenderData& render_data, const DataWriter<ImageBufferEvent>& writer) override;
    size_t scale_width() const { return scale_width_; }
    size_t scale_height() const { return scale_height_; }
private:
    size_t scale_width_, scale_height_;
};

// From<(&RendererConfig, &RenderConfig, &Image)> for Box<dyn Renderer>, renderer.rs:109-116.  Cpu and
// CpuPreview are the reference's own renderers and do not exist here: asking for them throws
// Configuration (there is no CPU fallback in this product).
std::unique_ptr<Renderer> make_renderer(RendererConfig which, const RenderConfig& config, const GpuConfig& gpu, const Image& image);

// ---- image_action/png.rs ----------------------------------------------------------------------
// SavePng::action: file name = upper-case SHA-256 of the RGBA bytes + ".png" inside image_output_dir
// (png.rs:36-41); returns the path written.  `explicit_path` overrides the name.
std::string save_png(const std::vector<uint8_t>& rgba, size_t width, size_t height, const std::string& image_output_dir,
                     const std::string& explicit_path = std::string());
std::string sha256_hex_upper(const uint8_t* data, size_t n);

}  // namespace racer
