// websplat_b200.hpp -- C++ host-side mirror of web-splat's render API above the C ABI (websplat_b200.h).
//
// The reference is compiled code (Rust) and its toolchain is absent from the image this repository was built in, so the
// host side above the ABI is mirrored here in C++ with the reference's names, argument meaning and error behaviour:
//   WGPUContext::new_instance        src/lib.rs:69            -> ws::Context
//   Aabb<f32>                        src/pointcloud.rs:398-463 -> ws::Aabb
//   PerspectiveProjection / Camera   src/camera.rs:7-152       -> ws::PerspectiveProjection, ws::PerspectiveCamera
//   focal2fov / fov2focal            src/camera.rs:236-242
//   SplattingArgs                    src/renderer.rs:587-599   -> ws::SplattingArgs (Option<T> = std::optional<T>)
//   PointCloud::new + getters        src/pointcloud.rs:99-349  -> ws::PointCloud (new_, from_ply, from_c3dgs)
//   GaussianRenderer                 src/renderer.rs:33-260    -> ws::GaussianRenderer (new_, prepare, render, ...)
//   SceneCamera / Scene              src/scene.rs:11-205       -> ws::SceneCamera, ws::Scene
// Errors: the reference panics / returns anyhow::Error; here every failing ABI call throws ws::Error (status + text).
// Header only; link against libwebsplat_b200.so.  (web-splat_b200/__init__.py is the same mirror in Python for the tests.)
#ifndef WEBSPLAT_B200_HPP
#define WEBSPLAT_B200_HPP

#include "websplat_b200.h"

#include <algorithm>
#include <array>
#include <cmath>
#include <cstring>
#include <map>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

namespace ws {

struct Error : std::runtime_error {
    ws_status status;
    Error(ws_status s, const std::string &what) : std::runtime_error(what), status(s) {}
};

inline void check(ws_status s)
{
    if (s == WS_OK) return;
    throw Error(s, std::string("websplat_b200: ") + ws_status_string(s) + " (status " + std::to_string(s) + "): " + ws_last_error());
}

/// WGPUContext::new_instance (src/lib.rs:69): one CUDA device.
class Context {
public:
    explicit Context(int cuda_device = 0) { check(ws_context_create(cuda_device, &h_)); }
    ~Context() { ws_context_destroy(h_); }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    ws_context *handle() const { return h_; }
    int device() const { return ws_context_device(h_); }
    int sm_count() const { return ws_context_sm_count(h_); }

private:
    ws_context *h_ = nullptr;
};

using Vec3 = std::array<float, 3>;
using Quat = std::array<float, 4>;   // (w, x, y, z) = cgmath Quaternion::new(w, xi, yj, zk)

/// Aabb<f32> (src/pointcloud.rs:398-463).
struct Aabb {
    Vec3 min{0, 0, 0}, max{0, 0, 0};
    ws_aabb c() const { ws_aabb b; std::memcpy(b.min, min.data(), 12); std::memcpy(b.max, max.data(), 12); return b; }
    static Aabb from_c(const ws_aabb &b) { Aabb a; std::memcpy(a.min.data(), b.min, 12); std::memcpy(a.max.data(), b.max, 12); return a; }
    Vec3 center() const { ws_aabb b = c(); Vec3 o; ws_aabb_center(&b, o.data()); return o; }
    float radius() const { ws_aabb b = c(); return ws_aabb_radius(&b); }
};

/// camera.rs:236-242 (f32 arithmetic like the reference).
inline float focal2fov(float focal, float pixels) { return 2.f * std::atan(pixels / (2.f * focal)); }
inline float fov2focal(float fov, float pixels) { return pixels / (2.f * std::tan(fov * 0.5f)); }

/// PerspectiveProjection (src/camera.rs:86-131); fov in radians.
struct PerspectiveProjection {
    float fovx = 0, fovy = 0, znear = 0.01f, zfar = 100.f, fov2view_ratio = 1.f;
    /// PerspectiveProjection::new (camera.rs:115-131)
    static PerspectiveProjection make(uint32_t width, uint32_t height, float fovx, float fovy, float znear, float zfar)
    {
        PerspectiveProjection p;
        const float vr = (float)width / (float)height, fr = fovx / fovy;
        p.fovx = fovx; p.fovy = fovy; p.znear = znear; p.zfar = zfar; p.fov2view_ratio = vr / fr;
        return p;
    }
};

/// PerspectiveCamera (src/camera.rs:7-35): Matrix3::from(rotation) is world->camera.
struct PerspectiveCamera {
    Vec3 position{0, 0, 0};
    Quat rotation{1, 0, 0, 0};
    PerspectiveProjection projection;
    /// fit_near_far (camera.rs:26-35)
    void fit_near_far(const Aabb &aabb)
    {
        ws_aabb b = aabb.c();
        ws_camera_fit_near_far(position.data(), &b, &projection.znear, &projection.zfar);
    }
};

/// SplattingArgs (src/renderer.rs:587-599), same fields, same Options.
struct SplattingArgs {
    PerspectiveCamera camera;
    std::array<uint32_t, 2> viewport{0, 0};
    float gaussian_scaling = 1.f;
    uint32_t max_sh_deg = 3;
    std::optional<bool> mip_splatting;
    std::optional<float> kernel_size;
    std::optional<Aabb> clipping_box;
    float walltime_secs = 100.f;                 // Duration::as_secs_f32 (renderer.rs:643)
    std::optional<Vec3> scene_center;            // ignored by the reference too (renderer.rs:644)
    std::optional<float> scene_extend;
    std::array<double, 4> background_color{0, 0, 0, 0};

    ws_splatting_args c() const
    {
        ws_splatting_args a;
        std::memset(&a, 0, sizeof a);
        std::memcpy(a.cam_position, camera.position.data(), 12);
        std::memcpy(a.cam_rotation_wxyz, camera.rotation.data(), 16);
        a.fovx = camera.projection.fovx; a.fovy = camera.projection.fovy;
        a.znear = camera.projection.znear; a.zfar = camera.projection.zfar;
        a.fov2view_ratio = camera.projection.fov2view_ratio;
        a.viewport[0] = viewport[0]; a.viewport[1] = viewport[1];
        a.gaussian_scaling = gaussian_scaling; a.max_sh_deg = max_sh_deg;
        if (mip_splatting) { a.has_mip_splatting = 1; a.mip_splatting = *mip_splatting ? 1 : 0; }
        if (kernel_size) { a.has_kernel_size = 1; a.kernel_size = *kernel_size; }
        if (clipping_box) { a.has_clipping_box = 1; a.clipping_box = clipping_box->c(); }
        a.walltime_secs = walltime_secs;
        if (scene_center) { a.has_scene_center = 1; std::memcpy(a.scene_center, scene_center->data(), 12); }
        if (scene_extend) { a.has_scene_extend = 1; a.scene_extend = *scene_extend; }
        for (int i = 0; i < 4; i++) a.background_color[i] = background_color[i];
        return a;
    }
};

/// PointCloud (src/pointcloud.rs:72-349).
class PointCloud {
public:
    /// PointCloud::new from the CPU byte buffers of a GenericGaussianPointCloud (io/mod.rs:27-42)
    static PointCloud new_(const Context &ctx, const ws_pointcloud_desc &desc) { PointCloud p; check(ws_pointcloud_create(ctx.handle(), &desc, &p.h_)); return p; }
    /// GenericGaussianPointCloud::load + PointCloud::new for a .ply image: the vertex conversion runs on the GPU
    static PointCloud from_ply(const Context &ctx, const void *file_bytes, size_t len) { PointCloud p; check(ws_pointcloud_create_from_ply(ctx.handle(), file_bytes, len, &p.h_)); return p; }
    /// the same for the decoded members of a compressed .npz
    static PointCloud from_c3dgs(const Context &ctx, const ws_c3dgs_arrays &arrays) { PointCloud p; check(ws_pointcloud_create_from_c3dgs(ctx.handle(), &arrays, &p.h_)); return p; }
    ~PointCloud() { ws_pointcloud_destroy(h_); }
    PointCloud(PointCloud &&o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    PointCloud &operator=(PointCloud &&o) noexcept { std::swap(h_, o.h_); return *this; }
    PointCloud(const PointCloud &) = delete;
    PointCloud &operator=(const PointCloud &) = delete;

    ws_pointcloud *handle() const { return h_; }
    uint32_t num_points() const { return ws_pointcloud_num_points(h_); }
    uint32_t sh_deg() const { return ws_pointcloud_sh_deg(h_); }
    bool compressed() const { return ws_pointcloud_compressed(h_) != 0; }
    Aabb bbox() const { ws_aabb b; check(ws_pointcloud_bbox(h_, &b)); return Aabb::from_c(b); }
    Vec3 center() const { Vec3 c; check(ws_pointcloud_center(h_, c.data())); return c; }
    std::optional<Vec3> up() const { Vec3 u; return ws_pointcloud_up(h_, u.data()) ? std::optional<Vec3>(u) : std::nullopt; }
    std::optional<bool> mip_splatting() const { int32_t v = 0; return ws_pointcloud_mip_splatting(h_, &v) ? std::optional<bool>(v != 0) : std::nullopt; }
    std::optional<float> dilation_kernel_size() const { float v = 0; return ws_pointcloud_dilation_kernel_size(h_, &v) ? std::optional<float>(v) : std::nullopt; }
    std::optional<Vec3> background_color() const { Vec3 c; return ws_pointcloud_background_color(h_, c.data()) ? std::optional<Vec3>(c) : std::nullopt; }

private:
    PointCloud() = default;
    ws_pointcloud *h_ = nullptr;
};

inline size_t bytes_per_pixel(ws_format f) { return f == WS_FORMAT_RGBA8_UNORM ? 4 : (f == WS_FORMAT_RGBA16_FLOAT ? 8 : 16); }

/// GaussianRenderer (src/renderer.rs:17-260).  Not re-entrant, like `&mut self` upstream.
class GaussianRenderer {
public:
    /// GaussianRenderer::new (renderer.rs:33): specialised on (format, sh_deg, compressed)
    static GaussianRenderer new_(const Context &ctx, ws_format color_format, uint32_t sh_deg, bool compressed)
    {
        GaussianRenderer r;
        check(ws_renderer_create(ctx.handle(), color_format, sh_deg, compressed ? 1 : 0, &r.h_));
        return r;
    }
    ~GaussianRenderer() { ws_renderer_destroy(h_); }
    GaussianRenderer(GaussianRenderer &&o) noexcept : h_(o.h_), views_(o.views_) { o.h_ = nullptr; }
    GaussianRenderer &operator=(GaussianRenderer &&o) noexcept { std::swap(h_, o.h_); std::swap(views_, o.views_); return *this; }
    GaussianRenderer(const GaussianRenderer &) = delete;
    GaussianRenderer &operator=(const GaussianRenderer &) = delete;

    /// prepare (renderer.rs:191): enqueues stage 1 + 2 on the caller's stream (cudaStream_t as void*).
    /// Throws ws::Error(WS_ERR_PAIR_OVERFLOW / WS_ERR_CUDA) ONCE when an EARLIER frame of this renderer turned out incomplete
    /// on the device (everything is asynchronous: the frame that overflowed could not fail its own call); nothing is enqueued
    /// by the throwing call, the next one proceeds.  stats() reports the status of the frame it synchronises.
    void prepare(void *stream, const PointCloud &pc, const SplattingArgs &render_settings)
    {
        const ws_splatting_args a = render_settings.c();
        check(ws_renderer_prepare(h_, pc.handle(), &a, stream));
    }
    /// render (renderer.rs:250) + the caller's LoadOp::Clear(clear): stage 3 into DEVICE memory
    void render(void *stream, const PointCloud &pc, void *target_device, size_t row_pitch, const std::array<double, 4> &clear)
    {
        check(ws_renderer_render(h_, pc.handle(), target_device, row_pitch, clear.data(), stream));
    }
    /// render + download_texture (bin/render.rs:187-246): the frame lands in host memory (asynchronously on `stream`)
    void render_to_host(void *stream, const PointCloud &pc, void *target_host, size_t row_pitch, const std::array<double, 4> &clear)
    {
        check(ws_renderer_render_to_host(h_, pc.handle(), target_host, row_pitch, clear.data(), stream));
    }
    /// num_visible_points (renderer.rs:170): blocking read-back of V
    uint32_t num_visible_points() { uint32_t v = 0; check(ws_renderer_num_visible_points(h_, &v)); return v; }
    /// batch of up to WS_MAX_VIEWS views of one cloud (one viewport): stage 1 + 2 for all of them
    void prepare_views(void *stream, const PointCloud &pc, const std::vector<SplattingArgs> &render_settings)
    {
        std::vector<ws_splatting_args> a;
        a.reserve(render_settings.size());
        for (const SplattingArgs &s : render_settings) a.push_back(s.c());
        check(ws_renderer_prepare_views(h_, pc.handle(), a.data(), (uint32_t)a.size(), stream));
        views_ = (uint32_t)a.size();
    }
    /// stage 3 of the batch into DEVICE memory: view v at target_device + v * view_stride
    void render_views(void *stream, const PointCloud &pc, void *target_device, size_t row_pitch, size_t view_stride,
                      const std::array<double, 4> &clear)
    {
        check(ws_renderer_render_views(h_, pc.handle(), target_device, row_pitch, view_stride, clear.data(), stream));
    }
    /// the same into host memory (asynchronously on `stream`)
    void render_views_to_host(void *stream, const PointCloud &pc, void *target_host, size_t row_pitch, size_t view_stride,
                              const std::array<double, 4> &clear)
    {
        check(ws_renderer_render_views_to_host(h_, pc.handle(), target_host, row_pitch, view_stride, clear.data(), stream));
    }
    /// per-view visible point counts of the last batch (blocking)
    std::vector<uint32_t> views_num_visible_points()
    {
        std::vector<uint32_t> v(views_);
        check(ws_renderer_views_num_visible_points(h_, v.data(), views_));
        return v;
    }
    /// the GPUStopwatch replacement: "preprocess" / "sorting" / "rasterization" (renderer.rs:220-239) in ms; synchronises
    ws_frame_stats stats() { ws_frame_stats s; check(ws_renderer_stats(h_, &s)); return s; }
    ws_format color_format() const { return ws_renderer_color_format(h_); }
    void set_timing(bool on) { check(ws_renderer_set_timing(h_, on ? 1 : 0)); }
    void set_pair_capacity(uint64_t max_pairs) { check(ws_renderer_set_pair_capacity(h_, max_pairs)); }
    ws_renderer *handle() const { return h_; }

private:
    GaussianRenderer() = default;
    ws_renderer *h_ = nullptr;
    uint32_t views_ = 0;       // views of the last prepare_views
};

// ---- dataset cameras (src/scene.rs) -----------------------------------------------------------------------------
enum class Split { Train, Test };
inline const char *to_string(Split s) { return s == Split::Train ? "train" : "test"; }

namespace detail {
/// cgmath 0.18 `Quaternion::from(Matrix3)`; m[r][c] is the math matrix (cgmath mat[c][r] = m[r][c]).
inline Quat quat_from_matrix(const float m[3][3])
{
    const float trace = (m[0][0] + m[1][1]) + m[2][2];
    const float half = 0.5f;
    float w, x, y, z;
    if (trace >= 0.f) {
        float s = std::sqrt(1.f + trace);
        w = half * s; s = half / s;
        x = (m[2][1] - m[1][2]) * s; y = (m[0][2] - m[2][0]) * s; z = (m[1][0] - m[0][1]) * s;
    } else if (m[0][0] > m[1][1] && m[0][0] > m[2][2]) {
        float s = std::sqrt((m[0][0] - m[1][1] - m[2][2]) + 1.f);
        x = half * s; s = half / s;
        y = (m[0][1] + m[1][0]) * s; z = (m[2][0] + m[0][2]) * s; w = (m[2][1] - m[1][2]) * s;
    } else if (m[1][1] > m[2][2]) {
        float s = std::sqrt((m[1][1] - m[0][0] - m[2][2]) + 1.f);
        y = half * s; s = half / s;
        z = (m[1][2] + m[2][1]) * s; x = (m[0][1] + m[1][0]) * s; w = (m[0][2] - m[2][0]) * s;
    } else {
        float s = std::sqrt((m[2][2] - m[0][0] - m[1][1]) + 1.f);
        z = half * s; s = half / s;
        x = (m[2][0] + m[0][2]) * s; y = (m[1][2] + m[2][1]) * s; w = (m[1][0] - m[0][1]) * s;
    }
    return Quat{w, x, y, z};
}
}  // namespace detail

/// SceneCamera (scene.rs:11-24): `rotation` keeps the file's nested arrays, each inner array one cgmath column.
struct SceneCamera {
    size_t id = 0;
    std::string img_name;
    uint32_t width = 0, height = 0;
    Vec3 position{0, 0, 0};
    float rotation[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    float fx = 0, fy = 0;
    Split split = Split::Train;

    /// `impl Into<PerspectiveCamera> for SceneCamera` (scene.rs:84-108)
    PerspectiveCamera into_perspective() const
    {
        const float fovx = focal2fov(fx, (float)width), fovy = focal2fov(fy, (float)height);
        float m[3][3];                                             // Matrix3::from([[f32;3];3]): inner arrays are columns
        for (int c = 0; c < 3; c++) for (int r = 0; r < 3; r++) m[r][c] = rotation[c][r];
        const double det = (double)m[0][0] * ((double)m[1][1] * m[2][2] - (double)m[1][2] * m[2][1])
                         - (double)m[0][1] * ((double)m[1][0] * m[2][2] - (double)m[1][2] * m[2][0])
                         + (double)m[0][2] * ((double)m[1][0] * m[2][1] - (double)m[1][1] * m[2][0]);
        if (det < 0.0) for (int c = 0; c < 3; c++) m[1][c] = -m[1][c];   // rot.x[1], rot.y[1], rot.z[1]
        PerspectiveCamera cam;
        cam.position = position;
        cam.rotation = detail::quat_from_matrix(m);
        cam.projection = PerspectiveProjection::make(width, height, fovx, fovy, 0.01f, 100.f);
        return cam;
    }
};

/// Scene (scene.rs:110-192): cameras by id (a later duplicate replaces the earlier one), every 8th entry is the test split.
class Scene {
public:
    explicit Scene(std::vector<SceneCamera> cameras)
    {
        float best = 0.f;                                          // max_distance (scene.rs:196-205)
        for (size_t i = 0; i < cameras.size(); i++)
            for (size_t j = i + 1; j < cameras.size(); j++) {
                float d2 = 0.f;
                for (int k = 0; k < 3; k++) { const float d = cameras[i].position[k] - cameras[j].position[k]; d2 += d * d; }
                best = std::max(best, d2);
            }
        extend_ = std::sqrt(best);
        for (auto &c : cameras) cameras_[c.id] = c;
    }
    /// from_json's split rule (scene.rs:140-147) for cameras parsed in file order
    static Scene from_file_order(std::vector<SceneCamera> cameras)
    {
        for (size_t i = 0; i < cameras.size(); i++) cameras[i].split = (i % 8 == 0) ? Split::Test : Split::Train;
        return Scene(std::move(cameras));
    }
    size_t num_cameras() const { return cameras_.size(); }
    float extend() const { return extend_; }
    std::optional<SceneCamera> camera(size_t id) const { auto it = cameras_.find(id); return it == cameras_.end() ? std::nullopt : std::optional<SceneCamera>(it->second); }
    /// cameras(split) sorted by id (scene.rs:160-172)
    std::vector<SceneCamera> cameras(std::optional<Split> split = std::nullopt) const
    {
        std::vector<SceneCamera> out;
        for (auto &kv : cameras_) if (!split || kv.second.split == *split) out.push_back(kv.second);   // std::map iterates in id order
        return out;
    }

private:
    std::map<size_t, SceneCamera> cameras_;
    float extend_ = 0.f;
};

/// download_texture's pixel conversion (bin/render.rs:234-240): clamp(f16 -> f32, 0, 1) * 255, truncated.
inline float half_to_float(uint16_t h)
{
    const uint32_t sign = (uint32_t)(h & 0x8000u) << 16, exp = (h >> 10) & 0x1fu, man = h & 0x3ffu;
    uint32_t bits;
    if (exp == 0) {
        if (man == 0) bits = sign;
        else { int e = -1; uint32_t m = man; do { e++; m <<= 1; } while (!(m & 0x400u)); bits = sign | ((uint32_t)(127 - 15 - e) << 23) | ((m & 0x3ffu) << 13); }
    } else if (exp == 31) bits = sign | 0x7f800000u | (man << 13);
    else bits = sign | ((exp + 112u) << 23) | (man << 13);
    float f; std::memcpy(&f, &bits, 4); return f;
}
inline uint8_t half_to_u8(uint16_t h)
{
    float f = half_to_float(h);
    if (!(f == f)) return 0;                                        // `NaN as u8` is 0 in Rust
    f = f < 0.f ? 0.f : (f > 1.f ? 1.f : f);
    return (uint8_t)(f * 255.f);
}

}  // namespace ws

#endif  // WEBSPLAT_B200_HPP
