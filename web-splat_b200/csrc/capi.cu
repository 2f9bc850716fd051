// capi.cu -- host side of libwebsplat_b200: the C ABI declared in include/websplat_b200.h.
//
// Mirrors the host logic of the reference's render API for the hot path:
//   PointCloud::new                     pointcloud.rs:99-199   -> ws_pointcloud_create
//   GaussianRenderer::new               renderer.rs:33-123     -> ws_renderer_create
//   GaussianRenderer::prepare           renderer.rs:191-248    -> ws_renderer_prepare
//     CameraUniform setters             renderer.rs:321-343
//     SplattingArgsUniform::from_args_and_pc   renderer.rs:620-651
//     GPURSSorter::create_sort_stuff    gpu_rs.rs:141-175 (lazy, on point-count change)
//   GaussianRenderer::render            renderer.rs:250-260    -> ws_renderer_render
//   GaussianRenderer::num_visible_points renderer.rs:170-189   -> ws_renderer_num_visible_points
//   GPUStopwatch                        utils.rs:26-134        -> ws_renderer_stats (CUDA events)
// There is no CPU fallback anywhere in this file: without a CUDA device every entry point
// that does work fails with WS_ERR_CUDA.
#include "../../include/websplat_b200.h"
#include "ws_device.cuh"
#include "ws_kernels.h"

#include <ctype.h>
#include <math.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>
#include <new>
#include <atomic>
#include <string>
#include <vector>

using namespace ws;

// ------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

static ws_status fail_cuda(cudaError_t e, const char *what)
{
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    g_last_error = buf;
    return (e == cudaErrorMemoryAllocation) ? WS_ERR_OUT_OF_MEMORY : WS_ERR_CUDA;
}
static ws_status fail(ws_status s, const char *what)
{
    g_last_error = what;
    return s;
}
#define CU(call)                                                         \
    do {                                                                 \
        cudaError_t e__ = (call);                                        \
        if (e__ != cudaSuccess) return fail_cuda(e__, #call);            \
    } while (0)

extern "C" const char *ws_status_string(ws_status s)
{
    switch (s) {
    case WS_OK: return "ok";
    case WS_ERR_INVALID_ARGUMENT: return "invalid argument";
    case WS_ERR_CUDA: return "CUDA error / no usable CUDA device";
    case WS_ERR_OUT_OF_MEMORY: return "out of device memory";
    case WS_ERR_PAIR_OVERFLOW: return "(tile, splat) pair capacity exceeded";
    case WS_ERR_NOT_PREPARED: return "render() called without prepare()";
    case WS_ERR_UNSUPPORTED: return "unsupported";
    case WS_ERR_MISMATCH: return "point cloud does not match the renderer specialisation";
    default: return "unknown status";
    }
}
extern "C" const char *ws_last_error(void) { return g_last_error.c_str(); }
extern "C" const char *ws_version(void) { return "websplat_b200 0.1 (sm_100a)"; }

// ------------------------------------------------------------------------------------
struct ws_context {
    int device;
    int sm_count;
    int cc_major, cc_minor;
};

extern "C" ws_status ws_context_create(int cuda_device, ws_context **out)
{
    if (!out) return fail(WS_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return fail_cuda(e, "cudaGetDeviceCount");
    if (count <= 0) return fail(WS_ERR_CUDA, "no CUDA device");
    if (cuda_device < 0 || cuda_device >= count) return fail(WS_ERR_INVALID_ARGUMENT, "cuda_device out of range");
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, cuda_device));
    if (prop.major != 10) return fail(WS_ERR_CUDA, "device is not compute capability 10.x (library is built for sm_100a only)");
    CU(cudaSetDevice(cuda_device));
    ws_context *c = new (std::nothrow) ws_context();
    if (!c) return fail(WS_ERR_OUT_OF_MEMORY, "host allocation failed");
    c->device = cuda_device;
    c->sm_count = prop.multiProcessorCount;
    c->cc_major = prop.major; c->cc_minor = prop.minor;
    *out = c;
    return WS_OK;
}
extern "C" void ws_context_destroy(ws_context *ctx) { delete ctx; }
extern "C" int ws_context_device(const ws_context *ctx) { return ctx ? ctx->device : -1; }
extern "C" int ws_context_sm_count(const ws_context *ctx) { return ctx ? ctx->sm_count : 0; }

// ------------------------------------------------------------------------------------
// camera helpers
extern "C" void ws_aabb_center(const ws_aabb *b, float out[3])
{
    for (int i = 0; i < 3; i++) out[i] = (b->min[i] + b->max[i]) * 0.5f;     // Point3::midpoint
}
extern "C" float ws_aabb_radius(const ws_aabb *b)
{
    float r2 = 0.f;
    for (int i = 0; i < 3; i++) { float t = b->max[i] - b->min[i]; r2 = r2 + t * t; }
    return sqrtf(r2) / 2.0f;                                                  // min.distance(max) / 2
}
extern "C" void ws_camera_fit_near_far(const float position[3], const ws_aabb *aabb, float *znear, float *zfar)
{
    // camera.rs:26-35
    float c[3]; ws_aabb_center(aabb, c);
    const float radius = ws_aabb_radius(aabb);
    float d2 = 0.f;
    for (int i = 0; i < 3; i++) { float t = c[i] - position[i]; d2 = d2 + t * t; }
    const float distance = sqrtf(d2);
    const float zf = distance + radius;
    float zn = distance - radius;
    const float lo = zf / 1000.f;
    if (!(zn > lo)) zn = lo;
    *zfar = zf; *znear = zn;
}

// CameraUniform::set_camera / set_viewport / set_focal, renderer.rs:136-141,321-343;
// world2view camera.rs:207-214 (closed form [R | -R t]); build_proj camera.rs:216-234.
static void build_camera_uniform(const ws_splatting_args *a, CameraUniform *u)
{
    const float s = a->cam_rotation_wxyz[0], x = a->cam_rotation_wxyz[1], y = a->cam_rotation_wxyz[2], z = a->cam_rotation_wxyz[3];
    const float x2 = x + x, y2 = y + y, z2 = z + z;
    const float xx2 = x2 * x, xy2 = x2 * y, xz2 = x2 * z, yy2 = y2 * y, yz2 = y2 * z, zz2 = z2 * z;
    const float sy2 = y2 * s, sz2 = z2 * s, sx2 = x2 * s;
    float R[3][3];   // [column][row], cgmath Matrix3::from(Quaternion)
    R[0][0] = 1.f - yy2 - zz2; R[0][1] = xy2 + sz2;       R[0][2] = xz2 - sy2;
    R[1][0] = xy2 - sz2;       R[1][1] = 1.f - xx2 - zz2; R[1][2] = yz2 + sx2;
    R[2][0] = xz2 + sy2;       R[2][1] = yz2 - sx2;       R[2][2] = 1.f - xx2 - yy2;
    memset(u, 0, sizeof *u);
    const float *t = a->cam_position;
    for (int c = 0; c < 3; c++)
        for (int r = 0; r < 3; r++) {
            u->view[c * 4 + r] = R[c][r];
            u->view_inv[r * 4 + c] = R[c][r];
        }
    for (int r = 0; r < 3; r++) {
        float acc = R[0][r] * t[0];
        acc = acc + R[1][r] * t[1];
        acc = acc + R[2][r] * t[2];
        u->view[12 + r] = -acc;
        u->view_inv[12 + r] = t[r];
    }
    u->view[15] = 1.f; u->view_inv[15] = 1.f;

    const float znear = a->znear, zfar = a->zfar;
    const float thy = tanf(a->fovy / 2.f), thx = tanf(a->fovx / 2.f);
    const float top = thy * znear, bottom = -top, right = thx * znear, left = -right;
    const float p00 = 2.0f * znear / (right - left);
    const float p11 = 2.0f * znear / (top - bottom);
    const float p02 = (right + left) / (right - left);
    const float p12 = (top + bottom) / (top - bottom);
    const float p22 = zfar / (zfar - znear);
    const float p23 = -(zfar * znear) / (zfar - znear);
    float P[16]; memset(P, 0, sizeof P);
    P[0] = p00; P[5] = p11; P[8] = p02; P[9] = p12; P[10] = p22; P[11] = 1.f; P[14] = p23;
    for (int c = 0; c < 4; c++)
        for (int r = 0; r < 4; r++) u->proj[c * 4 + r] = (r == 1) ? -P[c * 4 + r] : P[c * 4 + r];   // VIEWPORT_Y_FLIP * P
    u->proj_inv[0] = 1.f / p00; u->proj_inv[5] = 1.f / p11;
    u->proj_inv[12] = p02 / p00; u->proj_inv[13] = p12 / p11; u->proj_inv[14] = 1.f;
    u->proj_inv[11] = 1.f / p23; u->proj_inv[15] = -p22 / p23;
    u->viewport[0] = (float)a->viewport[0]; u->viewport[1] = (float)a->viewport[1];
    u->focal[0] = (float)a->viewport[0] / (2.f * tanf(a->fovx * 0.5f));
    u->focal[1] = (float)a->viewport[1] / (2.f * tanf(a->fovy * 0.5f));
}

// ------------------------------------------------------------------------------------
static uint64_t next_generation()
{
    static std::atomic<uint64_t> g{1};
    return g.fetch_add(1, std::memory_order_relaxed);
}

struct ws_pointcloud {
    ws_context *ctx;
    uint32_t n, sh_deg;
    bool compressed;
    uint8_t *d_gaussians = nullptr, *d_sh = nullptr, *d_covars = nullptr;
    float *d_xyz = nullptr;        // position plane (derived from the records at upload) for the count kernel
    Quant4 quant;
    ws_aabb aabb;
    float center[3];
    int32_t has_up; float up[3];
    int32_t has_mip, mip;
    int32_t has_kernel; float kernel;
    int32_t has_bg; float bg[3];
    size_t sh_bytes = 0;           // bytes of SH payload in d_sh (read-back)
    uint32_t num_covars = 0;
    uint64_t generation = next_generation();   // identity of THIS cloud in CUDA-graph cache keys (a freed cloud's address may be reused)
};

extern "C" void ws_pointcloud_destroy(ws_pointcloud *pc)
{
    if (!pc) return;
    cudaSetDevice(pc->ctx->device);
    cudaFree(pc->d_gaussians); cudaFree(pc->d_sh); cudaFree(pc->d_covars); cudaFree(pc->d_xyz);
    delete pc;
}

// load-time check of the two index fields of compressed records (ingest.cu: validate_compressed_kernel)
static ws_status validate_compressed_indices(ws_context *ctx, const uint8_t *d_gaussians, uint32_t n, uint32_t num_covars, uint32_t num_features)
{
    if (!n) return WS_OK;
    uint32_t *d_flag = nullptr, h_flag = 0;
    CU(cudaMalloc(&d_flag, 4));
    cudaError_t e = cudaMemset(d_flag, 0, 4);
    if (e == cudaSuccess) e = launch_validate_compressed(d_gaussians, n, num_covars, num_features, d_flag, ctx->sm_count * 8, 0);
    if (e == cudaSuccess) e = cudaMemcpy(&h_flag, d_flag, 4, cudaMemcpyDeviceToHost);
    cudaFree(d_flag);
    if (e != cudaSuccess) return fail_cuda(e, "validate_compressed_indices");
    if (h_flag) return fail(WS_ERR_INVALID_ARGUMENT, "compressed cloud: geometry_idx / sh_idx out of range of the codebooks");
    return WS_OK;
}

extern "C" ws_status ws_pointcloud_create(ws_context *ctx, const ws_pointcloud_desc *d, ws_pointcloud **out)
{
    if (!ctx || !d || !out) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    if (d->num_points > 0 && (!d->gaussians || !d->sh_coefs)) return fail(WS_ERR_INVALID_ARGUMENT, "gaussians / sh_coefs is NULL");
    if (d->num_points >= (1ull << 30)) return fail(WS_ERR_UNSUPPORTED, "more than 2^30 - 1 points");
    if (d->sh_deg > 3) return fail(WS_ERR_INVALID_ARGUMENT, "sh_deg > 3");
    if (d->compressed && (!d->covars || !d->quantization)) return fail(WS_ERR_INVALID_ARGUMENT, "compressed cloud needs covars + quantization");
    const uint32_t n = (uint32_t)d->num_points;
    const size_t rec = d->compressed ? 24u : 28u;
    if (!d->compressed && d->sh_bytes < (uint64_t)n * 96u) return fail(WS_ERR_INVALID_ARGUMENT, "sh_bytes < num_points * 96");
    CU(cudaSetDevice(ctx->device));
    ws_pointcloud *pc = new (std::nothrow) ws_pointcloud();
    if (!pc) return fail(WS_ERR_OUT_OF_MEMORY, "host allocation failed");
    pc->ctx = ctx; pc->n = n; pc->sh_deg = d->sh_deg; pc->compressed = d->compressed != 0;
    memset(&pc->quant, 0, sizeof pc->quant);
    if (d->quantization) memcpy(&pc->quant, d->quantization, sizeof pc->quant);
    pc->aabb = d->aabb;
    memcpy(pc->center, d->center, sizeof pc->center);
    pc->has_up = d->has_up; memcpy(pc->up, d->up, sizeof pc->up);
    pc->has_mip = d->has_mip_splatting; pc->mip = d->mip_splatting;
    pc->has_kernel = d->has_kernel_size; pc->kernel = d->kernel_size;
    pc->has_bg = d->has_background; memcpy(pc->bg, d->background_color, sizeof pc->bg);

    // records are padded to a whole 256-record partition so stage 1 can bulk-copy full partitions
    const size_t padded = ((size_t)n + 255u) / 256u * 256u;
    const size_t gbytes = (padded ? padded : 256u) * rec;
    cudaError_t e;
#define PC_CU(call) do { e = (call); if (e != cudaSuccess) { ws_status s__ = fail_cuda(e, #call); ws_pointcloud_destroy(pc); return s__; } } while (0)
    PC_CU(cudaMalloc(&pc->d_gaussians, gbytes));
    PC_CU(cudaMemset(pc->d_gaussians, 0, gbytes));
    if (n) PC_CU(cudaMemcpy(pc->d_gaussians, d->gaussians, (size_t)n * rec, cudaMemcpyHostToDevice));
    PC_CU(cudaMalloc(&pc->d_xyz, (size_t)(n ? n : 1) * 12u));
    if (n) PC_CU(cudaMemcpy2D(pc->d_xyz, 12, pc->d_gaussians, rec, 12, n, cudaMemcpyDeviceToDevice));   // xyz is the first 12 B of a record
    // raw SH is padded to whole 256-record partitions as well (stage 1 bulk-copies 24 KB blocks)
    size_t shb = d->sh_bytes ? (size_t)d->sh_bytes : 32u;
    if (!d->compressed && shb < (padded ? padded : 256u) * 96u) shb = (padded ? padded : 256u) * 96u;
    PC_CU(cudaMalloc(&pc->d_sh, shb + 32u));
    PC_CU(cudaMemset(pc->d_sh, 0, shb + 32u));
    if (d->sh_bytes) PC_CU(cudaMemcpy(pc->d_sh, d->sh_coefs, (size_t)d->sh_bytes, cudaMemcpyHostToDevice));
    pc->sh_bytes = d->compressed ? (size_t)d->sh_bytes : (size_t)n * 96u; pc->num_covars = (uint32_t)d->num_covars;
    if (d->compressed) {
        const size_t cb = (size_t)d->num_covars * 12u;
        PC_CU(cudaMalloc(&pc->d_covars, cb ? cb : 16u));
        if (cb) PC_CU(cudaMemcpy(pc->d_covars, d->covars, cb, cudaMemcpyHostToDevice));
    }
#undef PC_CU
    if (d->compressed) {
        const uint32_t per = (d->sh_deg + 1u) * (d->sh_deg + 1u) * 3u;
        const uint64_t nf = d->sh_bytes / per;
        ws_status vs = validate_compressed_indices(ctx, pc->d_gaussians, n, (uint32_t)d->num_covars, nf > 0xffffffffull ? 0xffffffffu : (uint32_t)nf);
        if (vs != WS_OK) { ws_pointcloud_destroy(pc); return vs; }
    }
    *out = pc;
    return WS_OK;
}

// ------------------------------------------------------------------------------------
// .ply ingest (SURVEY.md section 8(f) N1): PlyReader::new / read (io/ply.rs:28-48,165-195) +
// GenericGaussianPointCloud::new (io/mod.rs:63-105).  The header is parsed here; the vertex block is
// uploaded untouched and converted by ply.cu's kernel.
namespace {
struct PlyHeader {
    size_t data_offset = 0;
    uint64_t num_vertices = 0;
    uint32_t num_props = 0, num_f = 0;
    bool have_vertex = false, big_endian = false, ascii = false, non_float = false, layout_ok = true;
    int32_t has_mip = 0, mip = 0, has_kernel = 0, has_bg = 0;
    float kernel = 0.f, bg[3] = {0.f, 0.f, 0.f};
    bool bad_comment = false;
};
std::string trimmed(const std::string &t)
{
    size_t a = 0, b = t.size();
    while (a < b && isspace((unsigned char)t[a])) a++;
    while (b > a && isspace((unsigned char)t[b - 1])) b--;
    return t.substr(a, b - a);
}
std::string after_last_eq(const std::string &c)
{
    const size_t p = c.rfind('=');
    return trimmed(p == std::string::npos ? c : c.substr(p + 1));
}
bool parse_f32(const std::string &t, float *out)
{
    if (t.empty()) return false;
    char *end = nullptr;
    const float v = strtof(t.c_str(), &end);
    if (end == t.c_str() || *end != 0) return false;
    *out = v; return true;
}
// returns false when no complete header is found
bool parse_ply_header(const uint8_t *bytes, size_t len, PlyHeader *h)
{
    size_t pos = 0;
    int line_no = 0;
    std::string element;
    // the fixed property order read_line assumes (io/ply.rs:50-100)
    static const char *kHead[9] = {"x", "y", "z", "nx", "ny", "nz", "f_dc_0", "f_dc_1", "f_dc_2"};
    std::vector<std::string> props;
    while (pos < len) {
        size_t e = pos;
        while (e < len && bytes[e] != '\n') e++;
        if (e == len) return false;
        std::string line(reinterpret_cast<const char *>(bytes + pos), e - pos);
        pos = e + 1;
        if (!line.empty() && line.back() == '\r') line.pop_back();
        line_no++;
        if (line_no == 1) { if (trimmed(line) != "ply") return false; continue; }
        if (line == "end_header") { h->data_offset = pos; break; }
        if (line.rfind("format ", 0) == 0) {
            h->big_endian = line.find("binary_big_endian") != std::string::npos;
            h->ascii = line.find("ascii") != std::string::npos;
        } else if (line.rfind("comment", 0) == 0) {
            const std::string c = trimmed(line.substr(7));
            // first matching comment wins, like Iterator::find (io/ply.rs:121-160)
            if (c.find("mip") != std::string::npos && !h->has_mip && !h->bad_comment) {
                const std::string v = after_last_eq(c);
                if (v == "true") { h->has_mip = 1; h->mip = 1; }
                else if (v == "false") { h->has_mip = 1; h->mip = 0; }
                else h->bad_comment = true;
            }
            if (c.find("kernel_size") != std::string::npos && !h->has_kernel) {
                if (parse_f32(after_last_eq(c), &h->kernel)) h->has_kernel = 1; else h->bad_comment = true;
            }
            if (c.find("background_color") != std::string::npos && !h->has_bg) {
                // a malformed background only warns in the reference (io/ply.rs:37-39): leave it unset
                const std::string v = after_last_eq(c);
                float rgb[3]; int k = 0; size_t a = 0; bool ok = true;
                while (ok && a <= v.size()) {
                    size_t b = v.find(',', a);
                    if (b == std::string::npos) b = v.size();
                    float f;
                    if (!parse_f32(trimmed(v.substr(a, b - a)), &f)) ok = false;
                    else if (k < 3) rgb[k++] = f; else k++;
                    a = b + 1;
                }
                if (ok && k >= 3) { h->has_bg = 1; memcpy(h->bg, rgb, sizeof rgb); }
            }
        } else if (line.rfind("element ", 0) == 0) {
            char name[64]; unsigned long long cnt = 0;
            if (sscanf(line.c_str(), "element %63s %llu", name, &cnt) == 2) {
                element = name;
                if (element == "vertex") { h->have_vertex = true; h->num_vertices = cnt; }
            }
        } else if (line.rfind("property ", 0) == 0 && element == "vertex") {
            char type[64], name[128];
            if (sscanf(line.c_str(), "property %63s %127s", type, name) == 2) {
                if (strcmp(type, "float") != 0 && strcmp(type, "float32") != 0) h->non_float = true;
                props.push_back(name);
                if (strncmp(name, "f_", 2) == 0) h->num_f++;
            }
        }
    }
    if (!h->data_offset) return false;
    h->num_props = (uint32_t)props.size();
    for (size_t i = 0; i < 9 && i < props.size(); i++) if (props[i] != kHead[i]) h->layout_ok = false;
    if (props.size() >= 8) {
        static const char *kTail[8] = {"opacity", "scale_0", "scale_1", "scale_2", "rot_0", "rot_1", "rot_2", "rot_3"};
        for (size_t i = 0; i < 8; i++) if (props[props.size() - 8 + i] != kTail[i]) h->layout_ok = false;
    }
    return true;
}
inline float ord2f(uint32_t o) { uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o; float f; memcpy(&f, &u, 4); return f; }
}  // namespace

// GenericGaussianPointCloud::new / new_compressed statistics from the device reductions
static void finish_cloud_stats(ws_pointcloud *pc, uint32_t n, const double sums[9], const uint32_t mm[6], float box0)
{
    // bounding box: Aabb::zeroed() (raw, io/mod.rs:74-77) or Aabb::unit() (compressed, io/mod.rs:119-122)
    // grown by every point
    for (int d = 0; d < 3; d++) {
        const float lo = n ? ord2f(mm[d]) : -box0, hi = n ? ord2f(mm[3 + d]) : box0;
        pc->aabb.min[d] = fminf(-box0, lo); pc->aabb.max[d] = fmaxf(box0, hi);
    }
    // centroid + plane normal (plane_from_points, io/mod.rs:185-284) from f64 moments; the reference
    // accumulates in f32 in file order, so the last digits differ -- neither is on the render path
    // (centroid only feeds the intro reveal, `up` only the viewer's controller)
    const double inv_n = n ? 1.0 / (double)n : 0.0;
    const double cx = sums[0] * inv_n, cy = sums[1] * inv_n, cz = sums[2] * inv_n;
    pc->center[0] = (float)cx; pc->center[1] = (float)cy; pc->center[2] = (float)cz;
    if (!n) { const float qnan = nanf(""); pc->center[0] = pc->center[1] = pc->center[2] = qnan; }   // 0 * (1/0)
    pc->has_up = 0; pc->up[0] = pc->up[1] = pc->up[2] = 0.f;
    if (n >= 3) {
        const double xx = sums[3] * inv_n - cx * cx, xy = sums[4] * inv_n - cx * cy, xz = sums[5] * inv_n - cx * cz;
        const double yy = sums[6] * inv_n - cy * cy, yz = sums[7] * inv_n - cy * cz, zz = sums[8] * inv_n - cz * cz;
        double w[3] = {0, 0, 0};
        const double dets[3] = {yy * zz - yz * yz, xx * zz - xz * xz, xx * yy - xy * xy};
        const double axes[3][3] = {{dets[0], xz * yz - xy * zz, xy * yz - xz * yy},
                                   {xz * yz - xy * zz, dets[1], xy * xz - yz * xx},
                                   {xy * yz - xz * yy, xy * xz - yz * xx, dets[2]}};
        for (int k = 0; k < 3; k++) {
            double weight = dets[k] * dets[k];
            if (w[0] * axes[k][0] + w[1] * axes[k][1] + w[2] * axes[k][2] < 0.0) weight = -weight;
            for (int d = 0; d < 3; d++) w[d] += axes[k][d] * weight;
        }
        const double mag = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
        double nrm[3] = {w[0] / mag, w[1] / mag, w[2] / mag};
        if (nrm[1] < 0.0) for (int d = 0; d < 3; d++) nrm[d] = -nrm[d];
        if (isfinite(nrm[0]) && isfinite(nrm[1]) && isfinite(nrm[2])) {
            pc->has_up = 1;
            for (int d = 0; d < 3; d++) pc->up[d] = (float)nrm[d];
        }
    }
    {   // `if bbox.radius() < 10. { up = None; }` (io/mod.rs:87-89)
        const float dx = pc->aabb.max[0] - pc->aabb.min[0], dy = pc->aabb.max[1] - pc->aabb.min[1], dz = pc->aabb.max[2] - pc->aabb.min[2];
        if (sqrtf(dx * dx + dy * dy + dz * dz) / 2.f < 10.f) pc->has_up = 0;
    }
}

static ws_status check_ply_header(const uint8_t *bytes, uint64_t file_len, PlyHeader *h, uint32_t *sh_deg_out)
{
    if (!parse_ply_header(bytes, (size_t)file_len, h)) return fail(WS_ERR_INVALID_ARGUMENT, "not a .ply file / truncated header");
    if (!h->have_vertex) return fail(WS_ERR_INVALID_ARGUMENT, "missing element vertex");
    if (h->ascii) return fail(WS_ERR_UNSUPPORTED, "ascii ply format not supported");                 // io/ply.rs:181
    if (h->bad_comment) return fail(WS_ERR_INVALID_ARGUMENT, "could not parse a mip / kernel_size comment");
    if (h->num_f % 3u) return fail(WS_ERR_INVALID_ARGUMENT, "number of f_* properties is not a multiple of 3");
    const uint32_t ncoef = h->num_f / 3u;
    uint32_t root = 0;
    while (root * root < ncoef) root++;
    if (root * root != ncoef || root == 0) return fail(WS_ERR_INVALID_ARGUMENT, "number of sh coefficients cannot be mapped to sh degree");   // utils.rs:183-189
    if (root - 1u > 3) return fail(WS_ERR_UNSUPPORTED, "sh degree > 3");
    if (h->non_float || !h->layout_ok || h->num_props != 14u + 3u * ncoef)
        return fail(WS_ERR_UNSUPPORTED, "vertex properties are not the 3DGS layout x,y,z,nx,ny,nz,f_dc_*,f_rest_*,opacity,scale_*,rot_* (all float)");
    if (h->num_vertices >= (1ull << 30)) return fail(WS_ERR_UNSUPPORTED, "more than 2^30 - 1 points");
    if ((uint64_t)h->data_offset + h->num_vertices * (uint64_t)(h->num_props * 4u) > file_len) return fail(WS_ERR_INVALID_ARGUMENT, "vertex data truncated");
    *sh_deg_out = root - 1u;
    return WS_OK;
}

extern "C" ws_status ws_ply_probe(const void *file_bytes, uint64_t file_len, ws_ply_info *out)
{
    if (!out || (!file_bytes && file_len)) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    memset(out, 0, sizeof *out);
    PlyHeader h; uint32_t sh_deg = 0;
    const ws_status s = check_ply_header(static_cast<const uint8_t *>(file_bytes), file_len, &h, &sh_deg);
    if (s != WS_OK) return s;
    out->num_points = h.num_vertices; out->data_offset = h.data_offset;
    out->sh_deg = sh_deg; out->stride_bytes = h.num_props * 4u; out->big_endian = h.big_endian;
    out->has_mip_splatting = h.has_mip; out->mip_splatting = h.mip;
    out->has_kernel_size = h.has_kernel; out->kernel_size = h.kernel;
    out->has_background = h.has_bg; memcpy(out->background_color, h.bg, sizeof h.bg);
    return WS_OK;
}

extern "C" ws_status ws_pointcloud_create_from_ply(ws_context *ctx, const void *file_bytes, uint64_t file_len, ws_pointcloud **out)
{
    if (!ctx || !out || (!file_bytes && file_len)) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    const uint8_t *bytes = static_cast<const uint8_t *>(file_bytes);
    PlyHeader h; uint32_t sh_deg = 0;
    {
        const ws_status hs = check_ply_header(bytes, file_len, &h, &sh_deg);
        if (hs != WS_OK) return hs;
    }
    const uint32_t n = (uint32_t)h.num_vertices;
    const uint32_t stride = h.num_props * 4u;

    CU(cudaSetDevice(ctx->device));
    ws_pointcloud *pc = new (std::nothrow) ws_pointcloud();
    if (!pc) return fail(WS_ERR_OUT_OF_MEMORY, "host allocation failed");
    pc->ctx = ctx; pc->n = n; pc->sh_deg = sh_deg; pc->compressed = false;
    memset(&pc->quant, 0, sizeof pc->quant);
    pc->has_mip = h.has_mip; pc->mip = h.mip;
    pc->has_kernel = h.has_kernel; pc->kernel = h.kernel;
    pc->has_bg = h.has_bg; memcpy(pc->bg, h.bg, sizeof pc->bg);
    const size_t padded = ((size_t)n + 255u) / 256u * 256u;
    const size_t slots = padded ? padded : 256u;
    pc->sh_bytes = (size_t)n * 96u;
    uint8_t *d_raw = nullptr; double *d_sums = nullptr; uint32_t *d_mm = nullptr;
    cudaError_t e;
#define PLY_CU(call) do { e = (call); if (e != cudaSuccess) { ws_status s__ = fail_cuda(e, #call); cudaFree(d_raw); cudaFree(d_sums); ws_pointcloud_destroy(pc); return s__; } } while (0)
    PLY_CU(cudaMalloc(&pc->d_gaussians, slots * 28u));
    PLY_CU(cudaMemset(pc->d_gaussians, 0, slots * 28u));
    PLY_CU(cudaMalloc(&pc->d_sh, slots * 96u + 32u));
    PLY_CU(cudaMemset(pc->d_sh, 0, slots * 96u + 32u));
    PLY_CU(cudaMalloc(&pc->d_xyz, (size_t)(n ? n : 1) * 12u));
    PLY_CU(cudaMalloc(&d_sums, 9 * sizeof(double) + 8 * sizeof(uint32_t)));
    d_mm = reinterpret_cast<uint32_t *>(d_sums + 9);
    PLY_CU(cudaMemset(d_sums, 0, 9 * sizeof(double) + 8 * sizeof(uint32_t)));
    PLY_CU(cudaMemset(d_mm, 0xff, 3 * sizeof(uint32_t)));
    double sums[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t mm[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0, 0, 0};
    if (n) {
        PLY_CU(cudaMalloc(&d_raw, (size_t)n * stride));
        PLY_CU(cudaMemcpy(d_raw, bytes + h.data_offset, (size_t)n * stride, cudaMemcpyHostToDevice));
        PlyConvertArgs a;
        a.vertices = d_raw; a.n = n; a.stride_bytes = stride; a.sh_deg = sh_deg; a.big_endian = h.big_endian ? 1u : 0u;
        a.gaussians = pc->d_gaussians; a.sh_coefs = pc->d_sh; a.xyz = pc->d_xyz; a.sums = d_sums; a.minmax = d_mm;
        const unsigned want = (n + 255u) / 256u, cap = (unsigned)ctx->sm_count * 8u;
        PLY_CU(launch_ply_convert(a, (int)(want < cap ? want : cap), 0));
        PLY_CU(cudaMemcpy(sums, d_sums, sizeof sums, cudaMemcpyDeviceToHost));
        PLY_CU(cudaMemcpy(mm, d_mm, sizeof mm, cudaMemcpyDeviceToHost));
    }
#undef PLY_CU
    cudaFree(d_raw); cudaFree(d_sums);
    finish_cloud_stats(pc, n, sums, mm, 0.f);
    *out = pc;
    return WS_OK;
}

// .npz ingest (SURVEY.md section 8(f) N2): the array post-processing of NpzReader::read (io/npz.rs:58-225)
// + GenericGaussianPointCloud::new_compressed (io/mod.rs:107-150) on the GPU.
extern "C" ws_status ws_pointcloud_create_from_c3dgs(ws_context *ctx, const ws_c3dgs_arrays *d, ws_pointcloud **out)
{
    if (!ctx || !d || !out) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    if (d->sh_deg > 3) return fail(WS_ERR_INVALID_ARGUMENT, "sh_deg > 3");
    if (d->num_points >= (1ull << 30) || d->num_covars >= (1ull << 30) || d->num_features >= (1ull << 30))
        return fail(WS_ERR_UNSUPPORTED, "more than 2^30 - 1 entries");
    if (d->num_points && (!d->xyz || !d->opacity)) return fail(WS_ERR_INVALID_ARGUMENT, "xyz / opacity is NULL");
    if (d->num_covars && (!d->scaling || !d->rotation)) return fail(WS_ERR_INVALID_ARGUMENT, "scaling / rotation is NULL");
    if (d->num_features && (!d->features_dc || (d->sh_deg > 0 && !d->features_rest))) return fail(WS_ERR_INVALID_ARGUMENT, "features_dc / features_rest is NULL");
    // without index arrays entry i belongs to point i (io/npz.rs:179-186)
    if (!d->gaussian_indices && d->num_covars < d->num_points) return fail(WS_ERR_INVALID_ARGUMENT, "no gaussian_indices and fewer covariances than points");
    if (!d->feature_indices && d->num_features < d->num_points) return fail(WS_ERR_INVALID_ARGUMENT, "no feature_indices and fewer SH entries than points");
    const uint32_t n = (uint32_t)d->num_points, nc = (uint32_t)d->num_covars, nf = (uint32_t)d->num_features;
    const uint32_t per = (d->sh_deg + 1u) * (d->sh_deg + 1u) * 3u;

    CU(cudaSetDevice(ctx->device));
    ws_pointcloud *pc = new (std::nothrow) ws_pointcloud();
    if (!pc) return fail(WS_ERR_OUT_OF_MEMORY, "host allocation failed");
    pc->ctx = ctx; pc->n = n; pc->sh_deg = d->sh_deg; pc->compressed = true;
    memcpy(&pc->quant, &d->quantization, sizeof pc->quant);
    pc->has_mip = d->has_mip_splatting; pc->mip = d->mip_splatting;
    pc->has_kernel = d->has_kernel_size; pc->kernel = d->kernel_size;
    pc->has_bg = d->has_background; memcpy(pc->bg, d->background_color, sizeof pc->bg);
    const size_t padded = ((size_t)n + 255u) / 256u * 256u;
    const size_t slots = padded ? padded : 256u;
    // one staging allocation for all input arrays, 16-B aligned slices
    struct Slice { const void *src; size_t bytes, off; };
    Slice in[9] = {{d->xyz, (size_t)n * 6u, 0}, {d->opacity, (size_t)n, 0}, {d->scaling_factor, d->scaling_factor ? (size_t)n : 0u, 0},
                   {d->gaussian_indices, d->gaussian_indices ? (size_t)n * 4u : 0u, 0}, {d->feature_indices, d->feature_indices ? (size_t)n * 4u : 0u, 0},
                   {d->scaling, (size_t)nc * 3u, 0}, {d->rotation, (size_t)nc * 4u, 0},
                   {d->features_dc, (size_t)nf * 3u, 0}, {d->features_rest, (size_t)nf * (per - 3u), 0}};
    size_t total = 0;
    for (auto &sl : in) { sl.off = total; total += (sl.bytes + 15u) / 16u * 16u; }
    uint8_t *d_in = nullptr; double *d_sums = nullptr;
    cudaError_t e;
#define NPZ_CU(call) do { e = (call); if (e != cudaSuccess) { ws_status s__ = fail_cuda(e, #call); cudaFree(d_in); cudaFree(d_sums); ws_pointcloud_destroy(pc); return s__; } } while (0)
    NPZ_CU(cudaMalloc(&d_in, total ? total : 16u));
    for (auto &sl : in) if (sl.bytes) NPZ_CU(cudaMemcpy(d_in + sl.off, sl.src, sl.bytes, cudaMemcpyHostToDevice));
    NPZ_CU(cudaMalloc(&pc->d_gaussians, slots * 24u));
    NPZ_CU(cudaMemset(pc->d_gaussians, 0, slots * 24u));
    const size_t shb = (size_t)nf * per;
    NPZ_CU(cudaMalloc(&pc->d_sh, (shb ? shb : 32u) + 32u));
    NPZ_CU(cudaMemset(pc->d_sh, 0, (shb ? shb : 32u) + 32u));
    NPZ_CU(cudaMalloc(&pc->d_covars, nc ? (size_t)nc * 12u : 16u));
    NPZ_CU(cudaMalloc(&pc->d_xyz, (size_t)(n ? n : 1) * 12u));
    NPZ_CU(cudaMalloc(&d_sums, 9 * sizeof(double) + 8 * sizeof(uint32_t)));
    uint32_t *d_mm = reinterpret_cast<uint32_t *>(d_sums + 9);
    NPZ_CU(cudaMemset(d_sums, 0, 9 * sizeof(double) + 8 * sizeof(uint32_t)));
    NPZ_CU(cudaMemset(d_mm, 0xff, 3 * sizeof(uint32_t)));
    C3dgsArgs a;
    a.xyz_f16 = reinterpret_cast<const uint16_t *>(d_in + in[0].off);
    a.opacity = reinterpret_cast<const int8_t *>(d_in + in[1].off);
    a.scaling_factor = d->scaling_factor ? reinterpret_cast<const int8_t *>(d_in + in[2].off) : nullptr;
    a.gaussian_indices = d->gaussian_indices ? reinterpret_cast<const int32_t *>(d_in + in[3].off) : nullptr;
    a.feature_indices = d->feature_indices ? reinterpret_cast<const int32_t *>(d_in + in[4].off) : nullptr;
    a.scaling = reinterpret_cast<const int8_t *>(d_in + in[5].off);
    a.rotation = reinterpret_cast<const int8_t *>(d_in + in[6].off);
    a.features_dc = reinterpret_cast<const int8_t *>(d_in + in[7].off);
    a.features_rest = reinterpret_cast<const int8_t *>(d_in + in[8].off);
    a.n = n; a.num_covars = nc; a.num_features = nf; a.sh_deg = d->sh_deg;
    a.scaling_scale = d->scaling_scale; a.scaling_zero_point = (float)d->scaling_zero_point;       // `as f32`, io/npz.rs:66-72
    a.rotation_scale = d->rotation_scale; a.rotation_zero_point = (float)d->rotation_zero_point;
    a.gaussians = pc->d_gaussians; a.sh_out = reinterpret_cast<int8_t *>(pc->d_sh); a.covars = pc->d_covars; a.xyz = pc->d_xyz;
    a.sums = d_sums; a.minmax = d_mm;
    NPZ_CU(launch_c3dgs_convert(a, ctx->sm_count * 8, 0));
    double sums[9]; uint32_t mm[6];
    NPZ_CU(cudaMemcpy(sums, d_sums, sizeof sums, cudaMemcpyDeviceToHost));
    NPZ_CU(cudaMemcpy(mm, d_mm, sizeof mm, cudaMemcpyDeviceToHost));
#undef NPZ_CU
    cudaFree(d_in); cudaFree(d_sums);
    {   // gaussian_indices / feature_indices come from the file: reject out-of-range (incl. negative) entries
        ws_status vs = validate_compressed_indices(ctx, pc->d_gaussians, n, nc, nf);
        if (vs != WS_OK) { ws_pointcloud_destroy(pc); return vs; }
    }
    pc->sh_bytes = shb; pc->num_covars = nc;
    finish_cloud_stats(pc, n, sums, mm, 1.f);
    *out = pc;
    return WS_OK;
}

extern "C" uint64_t ws_pointcloud_buffer_bytes(const ws_pointcloud *pc, int32_t which)
{
    if (!pc) return 0;
    switch (which) {
    case 0: return (uint64_t)pc->n * (pc->compressed ? 24u : 28u);
    case 1: return pc->compressed ? pc->sh_bytes : (uint64_t)pc->n * 96u;
    case 2: return (uint64_t)pc->n * 12u;
    case 3: return (uint64_t)pc->num_covars * 12u;
    default: return 0;
    }
}

extern "C" ws_status ws_pointcloud_read(const ws_pointcloud *pc, int32_t which, void *dst, uint64_t dst_bytes)
{
    if (!pc || (!dst && dst_bytes)) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    const void *src = nullptr; size_t bytes = 0;
    switch (which) {
    case 0: src = pc->d_gaussians; bytes = (size_t)pc->n * (pc->compressed ? 24u : 28u); break;
    case 1: src = pc->d_sh; bytes = pc->compressed ? pc->sh_bytes : (size_t)pc->n * 96u; break;
    case 2: src = pc->d_xyz; bytes = (size_t)pc->n * 12u; break;
    case 3: src = pc->d_covars; bytes = (size_t)pc->num_covars * 12u; break;
    default: return fail(WS_ERR_INVALID_ARGUMENT, "unknown point-cloud buffer");
    }
    if (dst_bytes < bytes) return fail(WS_ERR_INVALID_ARGUMENT, "destination too small");
    CU(cudaSetDevice(pc->ctx->device));
    if (bytes) CU(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return WS_OK;
}

extern "C" uint32_t ws_pointcloud_num_points(const ws_pointcloud *pc) { return pc ? pc->n : 0; }
extern "C" uint32_t ws_pointcloud_sh_deg(const ws_pointcloud *pc) { return pc ? pc->sh_deg : 0; }
extern "C" int32_t ws_pointcloud_compressed(const ws_pointcloud *pc) { return pc ? (pc->compressed ? 1 : 0) : 0; }
extern "C" ws_status ws_pointcloud_bbox(const ws_pointcloud *pc, ws_aabb *out)
{
    if (!pc || !out) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = pc->aabb; return WS_OK;
}
extern "C" ws_status ws_pointcloud_center(const ws_pointcloud *pc, float out[3])
{
    if (!pc || !out) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    memcpy(out, pc->center, 12); return WS_OK;
}
extern "C" int32_t ws_pointcloud_up(const ws_pointcloud *pc, float out[3])
{
    if (!pc) return 0;
    if (pc->has_up && out) memcpy(out, pc->up, 12);
    return pc->has_up;
}
extern "C" int32_t ws_pointcloud_background_color(const ws_pointcloud *pc, float out[3])
{
    if (!pc) return 0;
    if (pc->has_bg && out) memcpy(out, pc->bg, 12);
    return pc->has_bg;
}
extern "C" int32_t ws_pointcloud_mip_splatting(const ws_pointcloud *pc, int32_t *out)
{
    if (!pc) return 0;
    if (pc->has_mip && out) *out = pc->mip;
    return pc->has_mip;
}
extern "C" int32_t ws_pointcloud_dilation_kernel_size(const ws_pointcloud *pc, float *out)
{
    if (!pc) return 0;
    if (pc->has_kernel && out) *out = pc->kernel;
    return pc->has_kernel;
}

// ------------------------------------------------------------------------------------
enum { EV_START = 0, EV_PRE, EV_DSORT, EV_BIN, EV_TSORT, EV_BLEND0, EV_BLEND1, EV_NEAR_BLEND, EV_BIN2, EV_TSORT2, EV_COUNT };
enum { TK_PRE = 0, TK_BIN = 1, TK_DSORT = 2, TK_TSORT = 6, TK_TSORT_FAR = 9 };

struct ShardState {
    uint32_t rank = 0, world = 0;              // world == 0: not sharded
    uint32_t width = 0, height = 0;
    uint32_t gated = 0;                        // several sharded frames in flight: flag waits in one-warp gate kernels
    uint32_t band_y0[9] = {};                  // tile-row bands: rank d owns rows [band_y0[d], band_y0[d+1])
    uint32_t recv_cap = 0, local_cap = 0;
    uint32_t *l_splats = nullptr, *l_keys = nullptr, *l_vals = nullptr; uint2 *l_rects = nullptr;   // stage-1 output of the local shard
    uint32_t *d_route = nullptr; size_t route_words = 0;
    uint32_t *part_band_counts = nullptr, *part_band_bases = nullptr, *hist_dummy = nullptr;
    uint32_t *peer_splats[8] = {}, *peer_keys[8] = {}; uint2 *peer_rects[8] = {};
    uint8_t *peer_frame[8][2] = {};            // every rank's two assembled-frame buffers (frame parity; only the root's are written)
    uint8_t *d_shard_frame[2] = {nullptr, nullptr}; size_t shard_frame_bytes = 0;
    ShardMailbox *d_mail = nullptr, *peer_mail[8] = {};   // rows / barrier / band flags written by the peers
    uint32_t epoch = 0;                        // host mirror of *d_epoch
    uint32_t *d_epoch = nullptr;               // frame number in device memory (advanced by the frame itself: graph replay)
    uint32_t *pending_signal = nullptr;        // set for the next band composite only
    // CUDA graphs of the single-call sharded frame (ws_renderer_shard_frame_to_root), one per frame-buffer parity
    cudaGraphExec_t frame_exec[2] = {nullptr, nullptr};
    struct { uint64_t pc_gen, buf_gen; uint32_t root, gated, bands[9]; float clear[4]; bool split; } frame_key[2] = {};
    bool opened[8] = {};
    bool imported = false;
    int phase = 0;
};

// What a captured prepare() graph depends on besides the sizes the kernels read from device memory
struct PrepKey {
    const ws_pointcloud *pc; uint64_t pc_gen, buf_gen; const void *gaussians, *scratch, *state; uint32_t n, K, W, H, pair_cap, n_cap; bool split;
    bool operator==(const PrepKey &o) const
    {
        return pc == o.pc && pc_gen == o.pc_gen && buf_gen == o.buf_gen && gaussians == o.gaussians && scratch == o.scratch &&
               state == o.state && n == o.n && K == o.K && W == o.W && H == o.H && pair_cap == o.pair_cap && n_cap == o.n_cap &&
               split == o.split;
    }
};

struct ws_renderer {
    ws_context *ctx;
    ws_format format;
    uint32_t sh_deg;
    bool compressed;
    bool timing = true;

    // capacities
    uint32_t n_cap = 0;            // points the sort buffers were created for (gpu_rs.rs:141)
    uint64_t pair_cap_req = 0;     // user request (0 = auto)
    uint32_t pair_cap = 0;
    uint32_t tiles_cap = 0;

    // device buffers
    FrameUniforms *d_uniforms = nullptr;
    uint8_t *d_scratch = nullptr; size_t scratch_bytes = 0;
    FrameCounters *d_counters = nullptr;
    uint32_t *d_hist_depth = nullptr, *d_hist_tile = nullptr;
    uint32_t *d_scan_pre = nullptr, *d_scan_bin = nullptr, *d_part_bases = nullptr, *d_bin_bases = nullptr;
    uint32_t *d_status_depth = nullptr, *d_status_tile = nullptr, *d_gstatus_depth = nullptr, *d_gstatus_tile = nullptr;
    uint32_t *d_splats = nullptr;
    uint32_t *d_keys[2] = {nullptr, nullptr}, *d_vals[2] = {nullptr, nullptr};
    uint2 *d_rects = nullptr;
    uint32_t *d_ptiles[2] = {nullptr, nullptr}, *d_pslots[2] = {nullptr, nullptr};
    uint2 *d_ranges = nullptr;
    void *d_frame = nullptr; size_t frame_bytes = 0;

    // launch geometry
    int grid_pre[2] = {0, 0}, grid_sort = 0, grid_bin = 0;     // grid_pre[batch]: single frames / batches of views

    // frame state
    FrameUniforms h_uniforms;
    bool prepared = false;
    bool rendered = false;
    int depth_passes = 4, tile_passes = 2;
    int depth_out = 0, tile_out = 0;       // which ping-pong buffer holds the sorted result
    cudaEvent_t ev[EV_COUNT] = {};
    bool ev_ok = false;
    cudaStream_t last_stream = nullptr;
    uint32_t last_n = 0;
    ShardState shard;
    // CUDA graph of one prepare() (clears + 14 kernels), replayed while (cloud, viewport, capacities) stay the same
    bool use_graphs = true;
    // occlusion split (two depth slabs, nearest first; DESIGN.md section 4)
    int split_mode = 2;                    // 0 off, 1 on, 2 auto (ws_renderer_set_occlusion_split)
    bool frame_split = false;              // the prepared frame was built split
    float4 *d_state = nullptr; size_t state_px = 0;   // per pixel {r, g, b, T} after the near slab
    uint8_t *d_tile_done = nullptr;        // per tile: saturated by the near slab
    uint32_t *d_keep4 = nullptr;           // far slab: one byte per splat, written by bin_count, read by bin_expand
    int tile_out_far = 0;
    cudaStream_t cap_stream = nullptr;
    // [batch]: a graph per mode, so a renderer that alternates single frames and batches never recaptures
    cudaGraphExec_t prep_exec[2] = {nullptr, nullptr};
    PrepKey prep_key[2] = {};
    // deferred frame status: render() copies {V, P, pair_overflow, error_flags} of its frame into a ring of pinned slots;
    // the NEXT prepare()/render() whose predecessor's copy has completed returns that frame's error once
    // (WS_ERR_PAIR_OVERFLOW / WS_ERR_CUDA) instead of WS_OK -- no synchronisation; ws_renderer_stats() consumes them too
    static constexpr int FLAG_SLOTS = 4;
    uint32_t *h_flags = nullptr;           // pinned, FLAG_SLOTS x 4 words
    cudaEvent_t ev_flags[FLAG_SLOTS] = {};
    bool flags_pending[FLAG_SLOTS] = {};
    int flag_next = 0;
    uint64_t buf_generation = 0;           // bumped whenever a buffer a captured graph points into is (re)allocated
    // d_uniforms holds 1 + WS_MAX_VIEWS blocks: [1 + v] = view v's own block, read by stage 1 (a single frame has K = 1
    // view), and [0] = the frame that stages 2-3 see, for a batch of views (ws_renderer_prepare_views) the "tall" frame
    // of K * tiles_y tile rows
    uint32_t views = 1;                    // views of the prepared frame
    bool batch = false;                    // the prepared frame is a batch (prepare_views)
    uint32_t *d_view_visible = nullptr;    // WS_MAX_VIEWS per-view survivor counts (in d_scratch)
    uint32_t *d_part_union = nullptr;      // per 256-Gaussian partition: survivors in any view (in d_scratch)
    FrameUniforms h_views[1 + WS_MAX_VIEWS];
};
static_assert(WS_MAX_VIEWS == MAX_VIEWS, "views per batch");

static void free_shard(ws_renderer *r);
static void free_sort_stuff(ws_renderer *r)
{
    cudaFree(r->d_scratch); r->d_scratch = nullptr;
    cudaFree(r->d_splats); r->d_splats = nullptr;
    for (int i = 0; i < 2; i++) {
        cudaFree(r->d_keys[i]); r->d_keys[i] = nullptr;
        cudaFree(r->d_vals[i]); r->d_vals[i] = nullptr;
        cudaFree(r->d_ptiles[i]); r->d_ptiles[i] = nullptr;
        cudaFree(r->d_pslots[i]); r->d_pslots[i] = nullptr;
    }
    cudaFree(r->d_rects); r->d_rects = nullptr;
    cudaFree(r->d_keep4); r->d_keep4 = nullptr;
    r->n_cap = 0; r->pair_cap = 0;
}

extern "C" void ws_renderer_destroy(ws_renderer *r)
{
    if (!r) return;
    cudaSetDevice(r->ctx->device);
    free_shard(r);
    free_sort_stuff(r);
    cudaFree(r->d_uniforms); cudaFree(r->d_ranges); cudaFree(r->d_frame); cudaFree(r->d_state); cudaFree(r->d_tile_done);
    if (r->ev_ok) for (int i = 0; i < EV_COUNT; i++) cudaEventDestroy(r->ev[i]);
    for (int i = 0; i < ws_renderer::FLAG_SLOTS; i++) if (r->ev_flags[i]) cudaEventDestroy(r->ev_flags[i]);
    if (r->h_flags) cudaFreeHost(r->h_flags);
    for (int i = 0; i < 2; i++) if (r->prep_exec[i]) cudaGraphExecDestroy(r->prep_exec[i]);
    if (r->cap_stream) cudaStreamDestroy(r->cap_stream);
    delete r;
}

extern "C" ws_status ws_renderer_create(ws_context *ctx, ws_format fmt, uint32_t sh_deg, int32_t compressed, ws_renderer **out)
{
    if (!ctx || !out) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    if ((int)fmt < 0 || (int)fmt > 2) return fail(WS_ERR_INVALID_ARGUMENT, "unknown color format");
    if (sh_deg > 3) return fail(WS_ERR_INVALID_ARGUMENT, "sh_deg > 3");
    CU(cudaSetDevice(ctx->device));
    ws_renderer *r = new (std::nothrow) ws_renderer();
    if (!r) return fail(WS_ERR_OUT_OF_MEMORY, "host allocation failed");
    r->ctx = ctx; r->format = fmt; r->sh_deg = sh_deg; r->compressed = compressed != 0;
    cudaError_t e = cudaMalloc(&r->d_uniforms, (1 + WS_MAX_VIEWS) * sizeof(FrameUniforms));
    if (e != cudaSuccess) { ws_status s = fail_cuda(e, "cudaMalloc uniforms"); ws_renderer_destroy(r); return s; }
    for (int i = 0; i < EV_COUNT; i++) {
        e = cudaEventCreate(&r->ev[i]);
        if (e != cudaSuccess) { ws_status s = fail_cuda(e, "cudaEventCreate"); ws_renderer_destroy(r); return s; }
    }
    r->ev_ok = true;
    e = cudaHostAlloc(reinterpret_cast<void **>(&r->h_flags), ws_renderer::FLAG_SLOTS * 16, cudaHostAllocDefault);
    for (int i = 0; i < ws_renderer::FLAG_SLOTS && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&r->ev_flags[i], cudaEventDisableTiming);
    if (e != cudaSuccess) { ws_status s = fail_cuda(e, "deferred-status slots"); ws_renderer_destroy(r); return s; }
    // persistent grids: one wave of resident CTAs
    for (int b = 0; b < 2; b++) r->grid_pre[b] = ctx->sm_count * preprocess_blocks_per_sm(r->compressed, b != 0);
    r->grid_sort = ctx->sm_count * sort_pass_blocks_per_sm();
    r->grid_bin = ctx->sm_count * binning_blocks_per_sm();
    {   // A/B knobs (profiles/): fewer resident CTAs per SM for the persistent kernels leave room for the other frame's kernels
        auto per_sm = [&](const char *name, int cur) { const char *e = getenv(name); const int k = e ? atoi(e) : 0; return (k >= 1 && k * ctx->sm_count < cur) ? k * ctx->sm_count : cur; };
        for (int b = 0; b < 2; b++) r->grid_pre[b] = per_sm("WS_PRE_CTAS_PER_SM", r->grid_pre[b]);
        r->grid_sort = per_sm("WS_SORT_CTAS_PER_SM", r->grid_sort);
        r->grid_bin = per_sm("WS_BIN_CTAS_PER_SM", r->grid_bin);
    }
    // 4 digit passes for both layouts: the compressed shader's "24-bit" key
    // (preprocess_compressed.wgsl:325) exceeds 0xffffff whenever clip.z < znear
    r->depth_passes = 4;
    memset(&r->h_uniforms, 0, sizeof r->h_uniforms);
    *out = r;
    return WS_OK;
}
extern "C" ws_format ws_renderer_color_format(const ws_renderer *r) { return r ? r->format : WS_FORMAT_RGBA8_UNORM; }

extern "C" ws_status ws_renderer_set_pair_capacity(ws_renderer *r, uint64_t max_pairs)
{
    if (!r) return fail(WS_ERR_INVALID_ARGUMENT, "NULL renderer");
    if (max_pairs >= (1ull << 30)) return fail(WS_ERR_UNSUPPORTED, "pair capacity must be < 2^30");
    r->pair_cap_req = max_pairs;
    return WS_OK;
}
extern "C" ws_status ws_renderer_set_timing(ws_renderer *r, int32_t enabled)
{
    if (!r) return fail(WS_ERR_INVALID_ARGUMENT, "NULL renderer");
    r->timing = enabled != 0;
    return WS_OK;
}
extern "C" ws_status ws_renderer_set_cuda_graphs(ws_renderer *r, int32_t enabled)
{
    if (!r) return fail(WS_ERR_INVALID_ARGUMENT, "NULL renderer");
    r->use_graphs = enabled != 0;
    return WS_OK;
}

// Occlusion split: 0 off, 1 on, negative = automatic (the default: on from 2 M points; the sharded paths never split).  Off = one binning + tile sort over all P pairs,
// which is what the pair-list read-backs (WS_BUF_PAIR_*, WS_BUF_TILE_RANGES) and num_pairs describe exactly.
extern "C" ws_status ws_renderer_set_occlusion_split(ws_renderer *r, int32_t enabled)
{
    if (!r) return fail(WS_ERR_INVALID_ARGUMENT, "NULL renderer");
    r->split_mode = enabled < 0 ? 2 : (enabled ? 1 : 0);
    return WS_OK;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// occlusion split: percentage of the depth-sorted splats that form the near slab (WS_SPLIT_NEAR_PCT; 0 / unset = the default, a quarter)
static uint32_t split_near_pct()
{
    static const uint32_t v = [] { const char *e = getenv("WS_SPLIT_NEAR_PCT"); const int p_ = e ? atoi(e) : 0; return (p_ >= 5 && p_ <= 95) ? (uint32_t)p_ : 0u; }();
    return v;
}

// compositor: cull against the box of still-unsaturated pixels (WS_ACTIVE_CULL=0 turns it off for A/B runs in profiles/)
static int active_cull_default()
{
    static const int v = [] { const char *e = getenv("WS_ACTIVE_CULL"); return (e && atoi(e) == 0) ? 0 : 1; }();
    return v;
}

// GPURSSorter::create_sort_stuff analogue (gpu_rs.rs:141-175, renderer.rs:200-211).  A batch of `views` views passes
// n = views x N: its automatic pair capacity, views x max(8 N, 1<<22), is what its views would get one by one.
static ws_status ensure_capacity(ws_renderer *r, uint32_t n, uint32_t tiles, uint32_t views = 1)
{
    uint64_t want_pairs = r->pair_cap_req;
    if (want_pairs == 0) {
        want_pairs = (uint64_t)n * 8u;
        if (want_pairs < (1ull << 22) * views) want_pairs = (1ull << 22) * views;
        if (want_pairs >= (1ull << 30)) want_pairs = (1ull << 30) - 1;
    }
    const uint32_t pair_cap = (uint32_t)want_pairs;
    if (!(r->d_scratch && r->n_cap == n && r->pair_cap == pair_cap)) {
        if (r->shard.world > 0 && r->d_scratch) return fail(WS_ERR_INVALID_ARGUMENT, "sharded renderer: capacities are fixed by ws_renderer_shard_configure");
        free_sort_stuff(r);
        const size_t nn = n ? n : 1;
        // + WS_MAX_VIEWS: a batch of K views of N points keeps K x ceil(N/256) partition counts, and n = K * N here
        const size_t parts256 = (nn + 255) / 256 + WS_MAX_VIEWS;
        const size_t sparts_n = (nn + SORT_PART - 1) / SORT_PART;
        const size_t sparts_p = ((size_t)pair_cap + SORT_PART - 1) / SORT_PART;
        size_t off = 0;
        const size_t o_counters = off; off = align_up(off + sizeof(FrameCounters), 256);
        const size_t o_hd = off; off = align_up(off + 4 * 256 * 4, 256);
        const size_t o_ht = off; off = align_up(off + 8 * 256 * 4, 256);      // 4 x 256 per slab
        const size_t o_sp = off; off = align_up(off + parts256 * 4, 256);
        const size_t o_sb = off; off = align_up(off + parts256 * 4, 256);
        const size_t o_pb = off; off = align_up(off + parts256 * 4, 256);
        const size_t o_bb = off; off = align_up(off + parts256 * 4, 256);
        const size_t o_un = off; off = align_up(off + parts256 * 4, 256);
        const size_t o_vv = off; off = align_up(off + WS_MAX_VIEWS * 4, 256);
        const size_t o_sd = off; off = align_up(off + 4 * sparts_n * 256 * 4, 256);
        const size_t o_st = off; off = align_up(off + 2 * 3 * sparts_p * 256 * 4, 256);     // x2: one set per depth slab
        const size_t gparts_n = (sparts_n + SORT_LB_GROUP - 1) / SORT_LB_GROUP, gparts_p = (sparts_p + SORT_LB_GROUP - 1) / SORT_LB_GROUP;
        const size_t o_gd = off; off = align_up(off + 4 * gparts_n * 256 * 4, 256);
        const size_t o_gt = off; off = align_up(off + 2 * 3 * gparts_p * 256 * 4, 256);
        CU(cudaMalloc(&r->d_scratch, off));
        r->scratch_bytes = off;
        r->d_counters = reinterpret_cast<FrameCounters *>(r->d_scratch + o_counters);
        r->d_hist_depth = reinterpret_cast<uint32_t *>(r->d_scratch + o_hd);
        r->d_hist_tile = reinterpret_cast<uint32_t *>(r->d_scratch + o_ht);
        r->d_scan_pre = reinterpret_cast<uint32_t *>(r->d_scratch + o_sp);
        r->d_scan_bin = reinterpret_cast<uint32_t *>(r->d_scratch + o_sb);
        r->d_part_bases = reinterpret_cast<uint32_t *>(r->d_scratch + o_pb);
        r->d_bin_bases = reinterpret_cast<uint32_t *>(r->d_scratch + o_bb);
        r->d_part_union = reinterpret_cast<uint32_t *>(r->d_scratch + o_un);
        r->d_view_visible = reinterpret_cast<uint32_t *>(r->d_scratch + o_vv);
        r->d_status_depth = reinterpret_cast<uint32_t *>(r->d_scratch + o_sd);
        r->d_status_tile = reinterpret_cast<uint32_t *>(r->d_scratch + o_st);
        r->d_gstatus_depth = reinterpret_cast<uint32_t *>(r->d_scratch + o_gd);
        r->d_gstatus_tile = reinterpret_cast<uint32_t *>(r->d_scratch + o_gt);
        CU(cudaMalloc(&r->d_splats, nn * 20));
        for (int i = 0; i < 2; i++) {
            CU(cudaMalloc(&r->d_keys[i], nn * 4));
            CU(cudaMalloc(&r->d_vals[i], nn * 4));
            CU(cudaMalloc(&r->d_ptiles[i], (size_t)pair_cap * 4));
            CU(cudaMalloc(&r->d_pslots[i], (size_t)pair_cap * 4));
        }
        CU(cudaMalloc(&r->d_rects, nn * 8));
        CU(cudaMalloc(&r->d_keep4, (nn + 2 * 1024 + 4) / 4 * 4 + 4096));   // one byte per far-slab splat (the far slab may be most of the cloud), rounded up to whole 1024-splat partitions
        r->n_cap = n; r->pair_cap = pair_cap;
        r->buf_generation = next_generation();
    }
    if (!r->d_ranges || r->tiles_cap < tiles) {
        cudaFree(r->d_ranges); r->d_ranges = nullptr;
        CU(cudaMalloc(&r->d_ranges, (size_t)(tiles ? tiles : 1) * 8 * 2));      // [tiles] near / only, [tiles] far slab
        cudaFree(r->d_tile_done); r->d_tile_done = nullptr;
        CU(cudaMalloc(&r->d_tile_done, (size_t)(tiles ? tiles : 1) + 64));     // + 64: bin_count packs it 32 bytes at a time with 128-bit loads
        r->tiles_cap = tiles;
        r->buf_generation = next_generation();
    }
    return WS_OK;
}

// SplattingArgsUniform::from_args_and_pc, renderer.rs:620-651
static void build_settings_uniform(const ws_splatting_args *a, const ws_pointcloud *pc, RenderSettings *s)
{
    memset(s, 0, sizeof *s);
    s->gaussian_scaling = a->gaussian_scaling;
    s->max_sh_deg = a->max_sh_deg;
    s->mip_splatting = a->has_mip_splatting ? (a->mip_splatting ? 1u : 0u) : ((pc->has_mip && pc->mip) ? 1u : 0u);
    s->kernel_size = a->has_kernel_size ? a->kernel_size : (pc->has_kernel ? pc->kernel : 0.3f /* DEFAULT_KERNEL_SIZE renderer.rs:601 */);
    const ws_aabb *cb = a->has_clipping_box ? &a->clipping_box : &pc->aabb;
    for (int i = 0; i < 3; i++) { s->clip_min[i] = cb->min[i]; s->clip_max[i] = cb->max[i]; }
    s->walltime = a->walltime_secs;
    for (int i = 0; i < 3; i++) s->center[i] = pc->center[i];         // args.scene_center is ignored (renderer.rs:644)
    const float rad = ws_aabb_radius(&pc->aabb);
    float ext = a->has_scene_extend ? a->scene_extend : rad;
    if (!(ext > rad)) ext = rad;                                       // .max(pc.bbox().radius())
    s->scene_extend = ext;
}

// Error of an EARLIER frame whose status copy has completed (see ws_renderer::h_flags); reported once.
static ws_status take_deferred_status(ws_renderer *r)
{
    ws_status st = WS_OK;
    for (int i = 0; i < ws_renderer::FLAG_SLOTS; i++) {
        if (!r->flags_pending[i] || cudaEventQuery(r->ev_flags[i]) != cudaSuccess) continue;
        r->flags_pending[i] = false;
        const uint32_t *f = r->h_flags + 4 * i;
        if (st == WS_OK && f[3]) st = WS_ERR_CUDA;
        if (st == WS_OK && f[2]) st = WS_ERR_PAIR_OVERFLOW;
    }
    cudaGetLastError();                                 // cudaErrorNotReady of a query is not an error
    if (st == WS_ERR_CUDA) return fail(st, "an earlier frame was incomplete: internal error flags set (look-back watchdog / receive capacity / peer wait)");
    if (st == WS_ERR_PAIR_OVERFLOW) return fail(st, "an earlier frame was incomplete: pair capacity exceeded; raise it with ws_renderer_set_pair_capacity");
    return WS_OK;
}

static ws_status validate_frame(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args)
{
    if (!r || !pc || !args) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (pc->compressed != r->compressed) return fail(WS_ERR_MISMATCH, "renderer/point cloud 'compressed' mismatch");
    if (r->compressed && pc->sh_deg != r->sh_deg) return fail(WS_ERR_MISMATCH, "compressed cloud sh_deg differs from the renderer's");
    if (args->viewport[0] == 0 || args->viewport[1] == 0) return fail(WS_ERR_INVALID_ARGUMENT, "empty viewport");
    if (args->viewport[0] > 16384 || args->viewport[1] > 16384) return fail(WS_ERR_UNSUPPORTED, "viewport larger than 16384");
    if (args->max_sh_deg > 3) return fail(WS_ERR_INVALID_ARGUMENT, "max_sh_deg > 3");
    if (r->compressed && args->max_sh_deg > r->sh_deg) return fail(WS_ERR_INVALID_ARGUMENT, "max_sh_deg exceeds the compressed cloud's degree");
    return WS_OK;
}

// Occlusion split on/off for this frame + the per-pixel state buffer it needs.  `points_here` = Gaussians this GPU
// depth-sorts (the whole cloud; total / world for sharded frames).  Automatic threshold: measured on one GPU cfg1
// (100 K points) -14 %, cfg2 (1 M) -2 %, cfg3 (6 M) +7 % -- the six extra launches and the state round trip pay off only
// when there are many pairs to save.
static ws_status decide_split(ws_renderer *r, uint64_t points_here, uint32_t W, uint32_t H, uint32_t views = 1)
{
    r->frame_split = r->split_mode == 1 || (r->split_mode == 2 && points_here >= 2000000u);
    if (r->frame_split) {
        const size_t px = (size_t)W * H * views;
        if (r->state_px < px) {
            cudaFree(r->d_state); r->d_state = nullptr; r->state_px = 0;
            CU(cudaMalloc(&r->d_state, px * sizeof(float4)));
            r->state_px = px;
            r->buf_generation = next_generation();
        }
    }
    return WS_OK;
}

static void build_frame_uniforms(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args, FrameUniforms *out);

// uniforms + per-frame clears (everything before stage 1) of a frame of K views that share the viewport (sharded
// frames: K = 1) and `capacity_points` splats.  A batch of K views is stacked into one "tall" frame of K * T tiles.
static ws_status begin_frame(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args, uint32_t K, bool batch,
                             uint32_t capacity_points, cudaStream_t stream, bool with_clears = true)
{
    const uint32_t W = args[0].viewport[0], H = args[0].viewport[1];
    const uint32_t tx = (W + TILE - 1) / TILE, ty = (H + TILE - 1) / TILE;
    const uint32_t tiles = tx * ty * K;              // < 2^23 for viewports up to 16384 and K <= 8
    r->prepared = false; r->rendered = false; r->batch = batch; r->views = K;
    ws_status st = ensure_capacity(r, capacity_points, tiles, K);
    if (st != WS_OK) return st;

    uint32_t max_deg = 0;
    for (uint32_t v = 0; v < K; v++) {
        build_frame_uniforms(r, pc, &args[v], &r->h_views[1 + v]);
        if (args[v].max_sh_deg > max_deg) max_deg = args[v].max_sh_deg;
    }
    FrameUniforms &T = r->h_views[0];                // stages 2-3: view 0's block with K * tiles_y tile rows
    T = r->h_views[1];
    T.tiles_y = ty * K;
    T.rs.max_sh_deg = max_deg;                       // read only by ws_renderer_stats (SH bytes of the batch)
    r->h_uniforms = T;
    r->tile_passes = (tiles > 65536u) ? 3 : ((tiles > 256u) ? 2 : 1);

    // one upload of the 1 + K blocks in front of the frame (pageable: staged before the call returns)
    CU(cudaMemcpyAsync(r->d_uniforms, r->h_views, (1 + K) * sizeof(FrameUniforms), cudaMemcpyHostToDevice, stream));
    if (with_clears) {
        CU(cudaMemsetAsync(r->d_scratch, 0, r->scratch_bytes, stream));
        CU(cudaMemsetAsync(r->d_ranges, 0xff, (size_t)r->tiles_cap * 8 * (r->frame_split ? 2 : 1), stream));    // {begin, ~end} identities for atomicMin (one set per depth slab)
    }
    return WS_OK;
}

static void build_frame_uniforms(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args, FrameUniforms *out)
{
    const uint32_t W = args->viewport[0], H = args->viewport[1];
    const uint32_t tx = (W + TILE - 1) / TILE, ty = (H + TILE - 1) / TILE;
    FrameUniforms &U = *out;
    build_camera_uniform(args, &U.cam);
    build_settings_uniform(args, pc, &U.rs);
    U.quant = pc->quant;
    U.width = W; U.height = H; U.tiles_x = tx; U.tiles_y = ty;
    U.num_points = pc->n; U.file_sh_deg = pc->sh_deg; U.pair_capacity = r->pair_cap; U._pad0 = 0;
    {   // per-frame constants of stage 1: one IEEE f32 division each, here instead of once per Gaussian
        volatile float one = 1.0f;                     // keep the host compiler from folding these into other precision
        U.inv_viewport[0] = one / U.cam.viewport[0]; U.inv_viewport[1] = one / U.cam.viewport[1];
        U.znear = -U.cam.proj[3 * 4 + 2] / U.cam.proj[2 * 4 + 2];
        U.zfar = -U.cam.proj[3 * 4 + 2] / (U.cam.proj[2 * 4 + 2] - 1.f);
        U.inv_scene_extend = one / U.rs.scene_extend;
        U._padf[0] = U._padf[1] = U._padf[2] = 0.f;
    }
}

// stage 2: depth passes on the V visible splats, tile binning, tile-id passes (+ ranges)
static ws_status enqueue_stage2(ws_renderer *r, cudaStream_t stream)
{
    {   // ---- stage 2a
        const size_t sparts_n = ((size_t)(r->n_cap ? r->n_cap : 1) + SORT_PART - 1) / SORT_PART;
        int src = 0;
        for (int p = 0; p < r->depth_passes; p++) {
            SortPassArgs a;
            a.keys_in = r->d_keys[src]; a.vals_in = r->d_vals[src];
            a.keys_out = r->d_keys[src ^ 1]; a.vals_out = r->d_vals[src ^ 1];
            a.n_ptr = &r->d_counters->num_visible; a.n_cap = r->n_cap;
            a.status = r->d_status_depth + (size_t)p * sparts_n * 256;
            a.gstatus = r->d_gstatus_depth + (size_t)p * ((sparts_n + SORT_LB_GROUP - 1) / SORT_LB_GROUP) * 256;
            a.ranges = nullptr;
            a.ticket = &r->d_counters->ticket[TK_DSORT + p];
            a.hist = r->d_hist_depth + p * 256;
            a.shift = 8u * (uint32_t)p;
            a.err = &r->d_counters->error_flags;
            CU(launch_sort_pass(a, r->grid_sort, stream));
            src ^= 1;
        }
        r->depth_out = src;
    }
    if (r->timing) CU(cudaEventRecord(r->ev[EV_DSORT], stream));
    // ---- stage 2b + 2c for one slab of the depth-sorted splats: expand into (tile, slot) pairs in depth order, then the
    //      tile-id passes on those pairs.  `half` selects the slab's private set of look-back status words, digit
    //      histograms, tickets and tile ranges (the pair buffers themselves are reused: the slabs run back to back).
    auto bin_and_tile_sort = [&](uint32_t slab, int half, int ev_bin, int ev_tsort, int *tile_out) -> ws_status {
        const size_t sparts_p = ((size_t)r->pair_cap + SORT_PART - 1) / SORT_PART;
        const size_t gparts_p = (sparts_p + SORT_LB_GROUP - 1) / SORT_LB_GROUP;
        // each slab has its own set of look-back status words (the second set starts after the 3 passes of the first)
        const size_t set_off = half ? 3 * sparts_p : 0, gset_off = half ? 3 * gparts_p : 0;
        const uint32_t cap = r->pair_cap;
        uint32_t *num_pairs = (slab == 1u) ? &r->d_counters->num_pairs_near : &r->d_counters->num_pairs;
        {
            BinningArgs a;
            a.sorted_slots = r->d_vals[r->depth_out]; a.rects = r->d_rects; a.uniforms = r->d_uniforms;
            a.counters = r->d_counters; a.pair_tiles = r->d_ptiles[0]; a.pair_slots = r->d_pslots[0];
            a.part_counts = r->d_scan_bin; a.part_bases = r->d_bin_bases; a.hist = r->d_hist_tile + half * 4 * 256;
            a.slab = slab; a.tile_done = (slab == 2u) ? r->d_tile_done : nullptr; a.pair_cap = cap; a.num_pairs_out = num_pairs;
            a.keep4 = r->d_keep4;
            a.num_tiles_hint = r->h_uniforms.tiles_x * r->h_uniforms.tiles_y; a.done_in_smem = 0;
            a.near_pct = split_near_pct();
            CU(launch_binning(a, r->ctx->sm_count * 8, r->grid_bin, stream));
        }
        if (r->timing) CU(cudaEventRecord(r->ev[ev_bin], stream));
        int src = 0;
        for (int p = 0; p < r->tile_passes; p++) {
            SortPassArgs a;
            a.keys_in = r->d_ptiles[src]; a.vals_in = r->d_pslots[src];
            a.keys_out = r->d_ptiles[src ^ 1]; a.vals_out = r->d_pslots[src ^ 1];
            a.n_ptr = num_pairs; a.n_cap = cap;
            a.status = r->d_status_tile + (set_off + (size_t)p * sparts_p) * 256;
            a.gstatus = r->d_gstatus_tile + (gset_off + (size_t)p * gparts_p) * 256;
            a.ranges = (p == r->tile_passes - 1) ? r->d_ranges + (half ? r->tiles_cap : 0) : nullptr;   // the last pass also emits the tile ranges
            // ... and nothing downstream reads the sorted tile ids (the compositor walks values + ranges): drop that store
            if (a.ranges && sort_pass_can_skip_keys()) a.keys_out = nullptr;
            a.ticket = &r->d_counters->ticket[(half ? TK_TSORT_FAR : TK_TSORT) + p];
            a.hist = r->d_hist_tile + half * 4 * 256 + p * 256;
            a.shift = 8u * (uint32_t)p;
            a.err = &r->d_counters->error_flags;
            CU(launch_sort_pass(a, r->grid_sort, stream));
            src ^= 1;
        }
        *tile_out = src;
        if (r->timing) CU(cudaEventRecord(r->ev[ev_tsort], stream));
        return WS_OK;
    };
    if (!r->frame_split) return bin_and_tile_sort(0u, 0, EV_BIN, EV_TSORT, &r->tile_out);

    // ---- occlusion split: near slab -> composite into per-pixel state + per-tile saturation -> far slab, whose
    //      binning drops every splat that only touches saturated tiles (most of them: a tile needs ~1/5 of its list)
    ws_status st = bin_and_tile_sort(1u, 0, EV_BIN, EV_TSORT, &r->tile_out);
    if (st != WS_OK) return st;
    {
        CompositeArgs a;
        memset(&a, 0, sizeof a);
        a.splats = r->d_splats; a.pair_slots = r->d_pslots[r->tile_out]; a.ranges = r->d_ranges;
        a.uniforms = r->d_uniforms; a.format = (int)r->format;
        a.mode = 1; a.state = r->d_state; a.tile_done = r->d_tile_done; a.active_cull = active_cull_default();
        // sharded frames: only this rank's band of tile rows (the received rectangles are clipped to it)
        const bool band = r->shard.world > 0;
        a.tile_y0 = band ? r->shard.band_y0[r->shard.rank] : 0u;
        const uint32_t rows = band ? r->shard.band_y0[r->shard.rank + 1] - r->shard.band_y0[r->shard.rank] : r->h_uniforms.tiles_y / r->views;
        if (rows) CU(launch_composite(a, r->h_uniforms.tiles_x, rows, stream, r->views));
    }
    if (r->timing) CU(cudaEventRecord(r->ev[EV_NEAR_BLEND], stream));
    return bin_and_tile_sort(2u, 1, EV_BIN2, EV_TSORT2, &r->tile_out_far);
}

// Stage-1 arguments of the frame begin_frame() set up: the view blocks d_uniforms[1..K] in, the depth sort's input out
static PreprocessArgs stage1_args(const ws_renderer *r, const ws_pointcloud *pc)
{
    PreprocessArgs a;
    a.gaussians = pc->d_gaussians; a.xyz = pc->d_xyz; a.sh_coefs = pc->d_sh; a.covars = pc->d_covars;
    a.uniforms = r->d_uniforms + 1;
    a.splats = r->d_splats; a.depth_keys = r->d_keys[0]; a.slot_vals = r->d_vals[0]; a.rects = r->d_rects;
    a.part_counts = r->d_scan_pre; a.part_bases = r->d_part_bases;
    a.hist = r->d_hist_depth; a.counters = r->d_counters;
    a.num_views = r->views; a.part_union = r->d_part_union; a.view_visible = r->d_view_visible;
    return a;
}

// Runs body() on `stream`, or -- with CUDA graphs on and timing off -- launches the graph in `exec`, first capturing it
// from body() when there is none or `same` is false (its key changed); *captured then tells the caller to store the
// new key.  `label` ends the error messages.
template <class Body>
static ws_status run_graph(ws_renderer *r, cudaGraphExec_t &exec, bool same, bool *captured, const char *label,
                           cudaStream_t stream, Body &&body)
{
    *captured = false;
    if (!r->use_graphs || r->timing) return body(stream);
    if (!exec || !same) {
        if (exec) { cudaGraphExecDestroy(exec); exec = nullptr; }
        if (!r->cap_stream) CU(cudaStreamCreateWithFlags(&r->cap_stream, cudaStreamNonBlocking));
        CU(cudaStreamBeginCapture(r->cap_stream, cudaStreamCaptureModeThreadLocal));
        ws_status st = body(r->cap_stream);
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaStreamEndCapture(r->cap_stream, &g);
        if (st != WS_OK) { if (g) cudaGraphDestroy(g); return st; }
        if (e != cudaSuccess) return fail_cuda(e, (std::string("cudaStreamEndCapture") + label).c_str());
        e = cudaGraphInstantiate(&exec, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) { exec = nullptr; return fail_cuda(e, (std::string("cudaGraphInstantiate") + label).c_str()); }
        *captured = true;
    }
    CU(cudaGraphLaunch(exec, stream));
    return WS_OK;
}

// Batches of views of one cloud (DESIGN.md "Batches of views").  The K views are stacked into one "tall" frame: tile
// (x, y) of view v is tile (v * tiles_y + y) * tiles_x + x.  Stage 1 runs once over the cloud for all views (view-major
// slots), stage 2 is the single-frame depth sort / binning / tile sort over the K * T tiles, and the compositor runs
// with gridDim.z = K.  Within each tile the order is (depth key, slot) with slots in Gaussian-index order, exactly as
// in a single frame, so every view is bit-identical to the same view rendered alone.
//
// ws_renderer_prepare is a single frame (K = 1, batch = false), ws_renderer_prepare_views a batch (batch = true, any
// K): a batch of one view still runs the batch instantiation of stage 1.
static ws_status prepare_frame(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args, uint32_t K, bool batch,
                               cudaStream_t stream)
{
    for (uint32_t v = 0; v < K; v++) {
        ws_status st = validate_frame(r, pc, &args[v]);
        if (st != WS_OK) return st;
        if (args[v].viewport[0] != args[0].viewport[0] || args[v].viewport[1] != args[0].viewport[1])
            return fail(WS_ERR_INVALID_ARGUMENT, "the views of a batch must share the viewport");
    }
    if (!batch && r->shard.world > 1) return fail(WS_ERR_INVALID_ARGUMENT, "renderer is configured for sharding: use ws_renderer_shard_begin/exchange/finish");
    if (batch && r->shard.world > 0) return fail(WS_ERR_INVALID_ARGUMENT, "batches of views are not supported on a sharded renderer");
    const uint64_t kn = (uint64_t)K * pc->n;         // a cloud has < 2^30 points: only a batch can reach the limit
    if (kn >= (1ull << 30)) return fail(WS_ERR_UNSUPPORTED, "num_views x num_points must be < 2^30 (30-bit look-back counts)");
    CU(cudaSetDevice(r->ctx->device));
    ws_status st = take_deferred_status(r);
    if (st != WS_OK) return st;
    const uint32_t W = args[0].viewport[0], H = args[0].viewport[1];
    st = decide_split(r, kn, W, H, K);
    if (st != WS_OK) return st;
    st = begin_frame(r, pc, args, K, batch, (uint32_t)kn, stream, /*with_clears=*/false);   // capacities may (re)allocate
    if (st != WS_OK) return st;

    // clears + stage 1 + stage 2
    auto body = [&](cudaStream_t q) -> ws_status {
        CU(cudaMemsetAsync(r->d_scratch, 0, r->scratch_bytes, q));
        CU(cudaMemsetAsync(r->d_ranges, 0xff, (size_t)r->tiles_cap * 8 * (r->frame_split ? 2 : 1), q));    // {begin, ~end} identities for atomicMin
        if (r->timing) CU(cudaEventRecord(r->ev[EV_START], q));
        CU(launch_preprocess(stage1_args(r, pc), r->compressed, batch, r->ctx->sm_count * 8, r->grid_pre[batch], q));
        if (r->timing) CU(cudaEventRecord(r->ev[EV_PRE], q));
        return enqueue_stage2(r, q);
    };
    // One CUDA graph per (cloud, viewport, views, capacities): 2 memsets + 14 kernels become one launch.  Every kernel
    // reads its sizes (N, V, P) from device memory, so the graph is independent of the frame's content.
    const PrepKey key = {pc, pc->generation, r->buf_generation, pc->d_gaussians, r->d_scratch, r->d_state,
                         pc->n, K, W, H, r->pair_cap, r->n_cap, r->frame_split};
    bool captured;
    st = run_graph(r, r->prep_exec[batch], r->prep_key[batch] == key, &captured, batch ? " (batch of views)" : "", stream, body);
    if (st != WS_OK) return st;
    if (captured) r->prep_key[batch] = key;
    r->prepared = true;
    r->last_stream = stream;
    r->last_n = pc->n;
    return WS_OK;
}

extern "C" ws_status ws_renderer_prepare(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args, void *cuda_stream)
{
    return prepare_frame(r, pc, args, 1, false, (cudaStream_t)cuda_stream);
}

extern "C" ws_status ws_renderer_prepare_views(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args,
                                               uint32_t num_views, void *cuda_stream)
{
    if (!r || !pc || !args) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (num_views == 0 || num_views > WS_MAX_VIEWS) return fail(WS_ERR_INVALID_ARGUMENT, "num_views must be in [1, WS_MAX_VIEWS]");
    return prepare_frame(r, pc, args, num_views, true, (cudaStream_t)cuda_stream);
}

// ------------------------------------------------------------------------------------
// Sharded (multi-GPU) frame: SURVEY.md 8(e), csrc/shard.cu.  One process per GPU; the host layer
// (torch.distributed / NCCL) moves the G x G count matrix and provides the barrier.
static void free_shard(ws_renderer *r)
{
    ShardState &s = r->shard;
    for (int p = 0; p < 8; p++) {
        if (s.opened[p]) {
            cudaIpcCloseMemHandle(s.peer_splats[p]); cudaIpcCloseMemHandle(s.peer_keys[p]); cudaIpcCloseMemHandle(s.peer_rects[p]);
            cudaIpcCloseMemHandle(s.peer_frame[p][0]); cudaIpcCloseMemHandle(s.peer_frame[p][1]); cudaIpcCloseMemHandle(s.peer_mail[p]);
            s.opened[p] = false;
        }
    }
    for (int i = 0; i < 2; i++) if (s.frame_exec[i]) cudaGraphExecDestroy(s.frame_exec[i]);
    cudaFree(s.l_splats); cudaFree(s.l_keys); cudaFree(s.l_vals); cudaFree(s.l_rects); cudaFree(s.d_route); cudaFree(s.d_shard_frame[0]); cudaFree(s.d_shard_frame[1]); cudaFree(s.d_mail); cudaFree(s.d_epoch);
    s = ShardState();
}

extern "C" ws_status ws_renderer_shard_configure(ws_renderer *r, uint32_t rank, uint32_t world, uint64_t total_points,
                                                 uint32_t local_points, uint32_t width, uint32_t height)
{
    if (!r) return fail(WS_ERR_INVALID_ARGUMENT, "NULL renderer");
    if (world < 1 || world > 8 || rank >= world) return fail(WS_ERR_INVALID_ARGUMENT, "need 1 <= world <= 8 and rank < world");
    if (total_points >= (1ull << 30) || width == 0 || height == 0) return fail(WS_ERR_INVALID_ARGUMENT, "bad total_points / viewport");
    CU(cudaSetDevice(r->ctx->device));
    free_shard(r);
    free_sort_stuff(r);
    ShardState &s = r->shard;
    s.rank = rank; s.world = world; s.width = width; s.height = height;
    s.recv_cap = (uint32_t)total_points;                 // worst case: every visible splat of every rank lands in one band
    s.local_cap = local_points ? local_points : 1;
    const uint32_t tx = (width + TILE - 1) / TILE, ty = (height + TILE - 1) / TILE;
    for (uint32_t d = 0; d <= world; d++) s.band_y0[d] = (uint32_t)(((uint64_t)ty * d) / world);   // contiguous tile-row bands
    // the pipeline buffers peers write into are allocated once and never move (IPC handles point at them)
    ws_status st = ensure_capacity(r, s.recv_cap, tx * ty);
    if (st != WS_OK) return st;
    const size_t nl = s.local_cap, parts = (nl + 1023) / 1024;          // routing partitions (shard.cu RT_PART)
    CU(cudaMalloc(&s.l_splats, nl * 20)); CU(cudaMalloc(&s.l_keys, nl * 4)); CU(cudaMalloc(&s.l_vals, nl * 4)); CU(cudaMalloc(&s.l_rects, nl * 8));
    s.route_words = parts * world * 2 + 4 * 256 + 16;
    CU(cudaMalloc(&s.d_route, s.route_words * 4));
    s.part_band_counts = s.d_route; s.part_band_bases = s.d_route + parts * world; s.hist_dummy = s.d_route + parts * world * 2;
    s.shard_frame_bytes = (size_t)width * height * (r->format == WS_FORMAT_RGBA8_UNORM ? 4 : (r->format == WS_FORMAT_RGBA16_FLOAT ? 8 : 16));
    CU(cudaMalloc(&s.d_shard_frame[0], s.shard_frame_bytes)); CU(cudaMalloc(&s.d_shard_frame[1], s.shard_frame_bytes));
    CU(cudaMalloc(&s.d_mail, sizeof(ShardMailbox)));
    CU(cudaMemset(s.d_mail, 0, sizeof(ShardMailbox)));
    CU(cudaMalloc(&s.d_epoch, 4));
    CU(cudaMemset(s.d_epoch, 0, 4));
    s.peer_splats[rank] = r->d_splats; s.peer_keys[rank] = r->d_keys[0]; s.peer_rects[rank] = r->d_rects;
    s.peer_frame[rank][0] = s.d_shard_frame[0]; s.peer_frame[rank][1] = s.d_shard_frame[1];
    s.peer_mail[rank] = s.d_mail;
    return WS_OK;
}

extern "C" ws_status ws_renderer_shard_export(ws_renderer *r, void *handles_6x64)
{
    void *handles_3x64 = handles_6x64;
    if (!r || !handles_3x64) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (r->shard.world < 1 || !r->d_splats) return fail(WS_ERR_INVALID_ARGUMENT, "call ws_renderer_shard_configure first");
    CU(cudaSetDevice(r->ctx->device));
    cudaIpcMemHandle_t h[6];
    CU(cudaIpcGetMemHandle(&h[0], r->d_splats)); CU(cudaIpcGetMemHandle(&h[1], r->d_keys[0])); CU(cudaIpcGetMemHandle(&h[2], r->d_rects));
    CU(cudaIpcGetMemHandle(&h[3], r->shard.d_shard_frame[0])); CU(cudaIpcGetMemHandle(&h[4], r->shard.d_shard_frame[1]));
    CU(cudaIpcGetMemHandle(&h[5], r->shard.d_mail));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handles_3x64, h, sizeof h);
    return WS_OK;
}

extern "C" ws_status ws_renderer_shard_import(ws_renderer *r, const void *all_handles)
{
    if (!r || !all_handles) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    ShardState &s = r->shard;
    if (s.world < 1) return fail(WS_ERR_INVALID_ARGUMENT, "call ws_renderer_shard_configure first");
    CU(cudaSetDevice(r->ctx->device));
    const cudaIpcMemHandle_t *h = static_cast<const cudaIpcMemHandle_t *>(all_handles);
    for (uint32_t p = 0; p < s.world; p++) {
        if (p == s.rank || s.opened[p]) continue;
        void *a = nullptr, *b = nullptr, *c = nullptr, *f = nullptr, *f1 = nullptr, *m = nullptr;
        CU(cudaIpcOpenMemHandle(&a, h[p * 6 + 0], cudaIpcMemLazyEnablePeerAccess));
        CU(cudaIpcOpenMemHandle(&b, h[p * 6 + 1], cudaIpcMemLazyEnablePeerAccess));
        CU(cudaIpcOpenMemHandle(&c, h[p * 6 + 2], cudaIpcMemLazyEnablePeerAccess));
        CU(cudaIpcOpenMemHandle(&f, h[p * 6 + 3], cudaIpcMemLazyEnablePeerAccess));
        CU(cudaIpcOpenMemHandle(&f1, h[p * 6 + 4], cudaIpcMemLazyEnablePeerAccess));
        CU(cudaIpcOpenMemHandle(&m, h[p * 6 + 5], cudaIpcMemLazyEnablePeerAccess));
        s.peer_mail[p] = static_cast<ShardMailbox *>(m);
        s.peer_splats[p] = static_cast<uint32_t *>(a); s.peer_keys[p] = static_cast<uint32_t *>(b); s.peer_rects[p] = static_cast<uint2 *>(c);
        s.peer_frame[p][0] = static_cast<uint8_t *>(f); s.peer_frame[p][1] = static_cast<uint8_t *>(f1);
        s.opened[p] = true;
    }
    s.imported = true;
    return WS_OK;
}

// Custom tile-row bands (cost-balanced partition of stages 2-3): band_y0[d] .. band_y0[d+1] are the tile rows of
// rank d.  Every rank must set the same boundaries, between frames.
extern "C" ws_status ws_renderer_shard_set_bands(ws_renderer *r, const uint32_t *band_y0, uint32_t count)
{
    if (!r || !band_y0) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    ShardState &s = r->shard;
    if (s.world < 1) return fail(WS_ERR_INVALID_ARGUMENT, "call ws_renderer_shard_configure first");
    const uint32_t ty = (s.height + TILE - 1) / TILE;
    if (count != s.world + 1 || band_y0[0] != 0 || band_y0[s.world] != ty) return fail(WS_ERR_INVALID_ARGUMENT, "need world + 1 boundaries from 0 to the number of tile rows");
    for (uint32_t d = 0; d < s.world; d++)
        if (band_y0[d + 1] <= band_y0[d]) return fail(WS_ERR_INVALID_ARGUMENT, "every rank needs at least one tile row");
    for (uint32_t d = 0; d <= s.world; d++) s.band_y0[d] = band_y0[d];
    return WS_OK;
}

extern "C" ws_status ws_renderer_shard_get_bands(const ws_renderer *r, uint32_t *band_y0, uint32_t count)
{
    if (!r || !band_y0) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    const ShardState &s = r->shard;
    if (s.world < 1 || count != s.world + 1) return fail(WS_ERR_INVALID_ARGUMENT, "not configured / need world + 1 entries");
    for (uint32_t d = 0; d <= s.world; d++) band_y0[d] = s.band_y0[d];
    return WS_OK;
}

// Several sharded frames in flight on this GPU (one renderer per frame slot, one stream each): move the peer-flag
// waits of ws_renderer_shard_frame_to_root out of the wide kernels into one-warp gate kernels.
extern "C" ws_status ws_renderer_shard_set_gated(ws_renderer *r, int32_t enabled)
{
    if (!r) return fail(WS_ERR_INVALID_ARGUMENT, "NULL renderer");
    r->shard.gated = enabled ? 1u : 0u;
    return WS_OK;
}

static void fill_route_args(ws_renderer *r, RouteArgs &a)
{
    ShardState &s = r->shard;
    a.l_splats = s.l_splats; a.l_keys = s.l_keys; a.l_rects = s.l_rects; a.counters = r->d_counters;
    a.world = s.world; a.rank = s.rank; a.gated = s.gated;
    for (int d = 0; d < 9; d++) a.band_y0[d] = s.band_y0[d < (int)s.world + 1 ? d : s.world];
    a.part_band_counts = s.part_band_counts; a.part_band_bases = s.part_band_bases;
    a.totals = nullptr; a.matrix = nullptr;
    for (int p = 0; p < 8; p++) { a.peer_splats[p] = s.peer_splats[p]; a.peer_keys[p] = s.peer_keys[p]; a.peer_rects[p] = s.peer_rects[p]; }
    a.recv_cap = s.recv_cap; a.err = &r->d_counters->error_flags;
    for (int p = 0; p < 8; p++) a.peer_mail[p] = nullptr;          // NCCL mode unless the caller fills these in
    a.epoch_ptr = s.d_epoch; a.done_counter = &r->d_counters->scatter_done;
}

extern "C" ws_status ws_renderer_shard_begin(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args,
                                             uint32_t *totals_row_device, void *cuda_stream)
{
    ws_status st = validate_frame(r, pc, args);
    if (st != WS_OK) return st;
    ShardState &s = r->shard;
    if (s.world < 1 || !totals_row_device) return fail(WS_ERR_INVALID_ARGUMENT, "renderer is not configured for sharding / NULL totals");
    if (s.world > 1 && !s.imported) return fail(WS_ERR_INVALID_ARGUMENT, "peer handles not imported");
    if (args->viewport[0] != s.width || args->viewport[1] != s.height) return fail(WS_ERR_INVALID_ARGUMENT, "viewport differs from ws_renderer_shard_configure");
    if (pc->n > s.local_cap) return fail(WS_ERR_INVALID_ARGUMENT, "local shard larger than configured");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(cudaSetDevice(r->ctx->device));
    r->frame_split = false;
    st = begin_frame(r, pc, args, 1, false, s.recv_cap, stream);
    if (st != WS_OK) return st;
    if (r->timing) CU(cudaEventRecord(r->ev[EV_START], stream));
    {   // ---- stage 1 on the local shard, into the local staging arrays
        PreprocessArgs a = stage1_args(r, pc);
        a.splats = s.l_splats; a.depth_keys = s.l_keys; a.slot_vals = s.l_vals; a.rects = s.l_rects;
        a.hist = s.hist_dummy;                                   // the consumer histograms the keys it RECEIVES
        CU(cudaMemsetAsync(s.hist_dummy, 0, 4 * 256 * 4, stream));
        CU(launch_preprocess(a, r->compressed, false, r->ctx->sm_count * 8, r->grid_pre[0], stream));
    }
    {   // ---- routing pass 1+2: how many local splats go to each band
        RouteArgs a; fill_route_args(r, a);
        a.totals = totals_row_device;
        CU(launch_route_count(a, r->ctx->sm_count * 8, stream));
    }
    if (r->timing) CU(cudaEventRecord(r->ev[EV_PRE], stream));
    r->last_stream = stream; r->last_n = pc->n;
    s.phase = 1;
    return WS_OK;
}

extern "C" ws_status ws_renderer_shard_exchange(ws_renderer *r, const uint32_t *matrix_device, void *cuda_stream)
{
    if (!r || !matrix_device) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    ShardState &s = r->shard;
    if (s.phase != 1) return fail(WS_ERR_NOT_PREPARED, "ws_renderer_shard_begin must precede exchange");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(cudaSetDevice(r->ctx->device));
    RouteArgs a; fill_route_args(r, a);
    a.matrix = matrix_device;
    CU(launch_route_scatter(a, r->ctx->sm_count * 8, stream));      // stores straight into the owners' buffers (NVLink)
    s.phase = 2;
    return WS_OK;
}

extern "C" ws_status ws_renderer_shard_finish(ws_renderer *r, const uint32_t *matrix_device, void *cuda_stream)
{
    if (!r || !matrix_device) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    ShardState &s = r->shard;
    if (s.phase != 2) return fail(WS_ERR_NOT_PREPARED, "ws_renderer_shard_exchange (and the cross-rank barrier) must precede finish");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(cudaSetDevice(r->ctx->device));
    CU(launch_shard_finish(matrix_device, s.world, s.rank, s.recv_cap, r->d_counters, r->d_vals[0], r->ctx->sm_count * 4, stream));
    CU(launch_sort_histogram(r->d_keys[0], &r->d_counters->num_visible, r->n_cap, r->d_hist_depth, r->depth_passes, r->ctx->sm_count * 4, stream));
    if (r->timing) CU(cudaEventRecord(r->ev[EV_PRE], stream));     // "preprocess" = stage 1 + exchange in sharded mode
    ws_status st = enqueue_stage2(r, stream);
    if (st != WS_OK) return st;
    r->prepared = true;
    r->last_stream = stream;
    s.phase = 0;
    return WS_OK;
}

static ws_status render_rows(ws_renderer *r, ws_pointcloud *pc, void *dst, size_t row_pitch, const double clear[4],
                             void *cuda_stream, uint32_t tile_y0, uint32_t tile_rows, size_t view_stride = 0);
static ws_status enqueue_composite(ws_renderer *r, void *dst, size_t row_pitch, const double clear[4], cudaStream_t stream,
                                   uint32_t tile_y0, uint32_t tile_rows, size_t view_stride = 0);
static ws_status enqueue_status_copy(ws_renderer *r, cudaStream_t stream);

// The whole sharded frame in ONE call and with NO host-side collective: the count rows, the barrier
// after the exchange and the "band has landed" signal are epoch flags that the kernels themselves
// write into the peers' mailboxes (release / acquire at system scope over NVLink).  The frame ends up
// assembled in rank `root`'s frame buffer (ws_renderer_shard_frame / _download); on the root the call
// also enqueues the wait for all bands.  Every rank must call it once per frame, in the same order.
extern "C" ws_status ws_renderer_shard_frame_to_root(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args,
                                                     uint32_t root, const double clear[4], void *cuda_stream)
{
    ws_status st = validate_frame(r, pc, args);
    if (st != WS_OK) return st;
    ShardState &s = r->shard;
    if (s.world < 1 || root >= s.world) return fail(WS_ERR_INVALID_ARGUMENT, "renderer is not configured for sharding / bad root");
    if (s.world > 1 && !s.imported) return fail(WS_ERR_INVALID_ARGUMENT, "peer handles not imported");
    if (args->viewport[0] != s.width || args->viewport[1] != s.height) return fail(WS_ERR_INVALID_ARGUMENT, "viewport differs from ws_renderer_shard_configure");
    if (pc->n > s.local_cap) return fail(WS_ERR_INVALID_ARGUMENT, "local shard larger than configured");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(cudaSetDevice(r->ctx->device));
    st = take_deferred_status(r);
    if (st != WS_OK) return st;
    // occlusion split inside the band (same bit-identical two-slab scheme as the single-GPU frame): automatic when this
    // rank's share of the cloud is large enough to pay for the extra launches (2 GPUs at cfg3: yes; 8 GPUs: no)
    st = decide_split(r, (uint64_t)s.recv_cap / s.world, s.width, s.height);
    if (st != WS_OK) return st;
    st = begin_frame(r, pc, args, 1, false, s.recv_cap, stream, /*with_clears=*/false);      // uniforms (an ordinary async copy in front of the frame)
    if (st != WS_OK) return st;
    const uint32_t rows = s.band_y0[s.rank + 1] - s.band_y0[s.rank];
    if (rows == 0 || s.band_y0[s.rank] * TILE >= s.height) return fail(WS_ERR_UNSUPPORTED, "a rank without tile rows (more ranks than tile rows) is not supported");
    const uint32_t par = (s.epoch + 1u) & 1u;           // parity of the frame buffer this frame fills (host mirror of the device epoch:
                                                        // committed below, once the frame -- whose first kernel advances the device word -- is enqueued)

    // everything of the frame that does not depend on the frame's content: clears, epoch, stage 1, routing + exchange,
    // stage 2, the band compositor (pixels into the root's frame of this parity), the root's wait for all bands
    auto body = [&](cudaStream_t q) -> ws_status {
        CU(cudaMemsetAsync(r->d_scratch, 0, r->scratch_bytes, q));
        CU(cudaMemsetAsync(r->d_ranges, 0xff, (size_t)r->tiles_cap * 8 * (r->frame_split ? 2 : 1), q));
        CU(cudaMemsetAsync(s.hist_dummy, 0, 4 * 256 * 4, q));
        CU(launch_epoch_advance(s.d_epoch, q));
        if (r->timing) CU(cudaEventRecord(r->ev[EV_START], q));
        {   // stage 1 on the local shard
            PreprocessArgs a = stage1_args(r, pc);
            a.splats = s.l_splats; a.depth_keys = s.l_keys; a.slot_vals = s.l_vals; a.rects = s.l_rects;
            a.hist = s.hist_dummy;
            CU(launch_preprocess(a, r->compressed, false, r->ctx->sm_count * 8, r->grid_pre[0], q));
        }
        RouteArgs ra; fill_route_args(r, ra);
        for (uint32_t p = 0; p < s.world; p++) ra.peer_mail[p] = s.peer_mail[p];
        CU(launch_route_count(ra, r->ctx->sm_count * 8, q));          // counts + scan; the row goes to every rank's mailbox
        CU(launch_route_scatter(ra, r->ctx->sm_count * 8, q));        // waits for all rows, stores the splats into the owners' buffers
        CU(launch_shard_finish_peer(ra, r->d_vals[0], r->d_keys[0], r->d_hist_depth, r->depth_passes, r->d_counters,
                                    r->ctx->sm_count * 4, q));        // waits for every rank's exchange flag
        if (r->timing) CU(cudaEventRecord(r->ev[EV_PRE], q));
        ws_status bs = enqueue_stage2(r, q);
        if (bs != WS_OK) return bs;
        // stage 3: pixels go straight into the root's frame; the last CTA raises this rank's band flag there
        const size_t pitch = s.shard_frame_bytes / s.height;
        s.pending_signal = &s.peer_mail[root]->flag_band[s.rank];
        bs = enqueue_composite(r, s.peer_frame[root][par] + (size_t)(s.band_y0[s.rank] * TILE) * pitch, pitch, clear, q, s.band_y0[s.rank], rows);
        if (bs != WS_OK) return bs;
        if (s.rank == root) CU(launch_wait_bands(s.d_mail, s.world, s.d_epoch, &r->d_counters->error_flags, q));
        return WS_OK;
    };

    // One CUDA graph per frame-buffer parity: ~25 launches + 3 clears become one launch (host: ~200 -> ~60 us per
    // frame and rank; device: no launch gaps between the latency-bound kernels of a 1/8 share of the frame).
    auto &k = s.frame_key[par];
    bool same = k.pc_gen == pc->generation && k.buf_gen == r->buf_generation && k.root == root && k.gated == s.gated &&
                k.split == r->frame_split;
    for (int i = 0; i < 9 && same; i++) same = k.bands[i] == s.band_y0[i];
    for (int i = 0; i < 4 && same; i++) same = k.clear[i] == (clear ? (float)clear[i] : 0.f);
    bool captured;
    st = run_graph(r, s.frame_exec[par], same, &captured, " (sharded frame)", stream, body);
    if (st != WS_OK) return st;
    if (captured) {
        k.pc_gen = pc->generation; k.buf_gen = r->buf_generation; k.root = root; k.gated = s.gated; k.split = r->frame_split;
        for (int i = 0; i < 9; i++) k.bands[i] = s.band_y0[i];
        for (int i = 0; i < 4; i++) k.clear[i] = clear ? (float)clear[i] : 0.f;
    }
    s.epoch += 1;
    st = enqueue_status_copy(r, stream);
    if (st != WS_OK) return st;
    r->prepared = true; r->rendered = true; r->last_stream = stream; r->last_n = pc->n;
    return WS_OK;
}

extern "C" ws_status ws_renderer_shard_band(const ws_renderer *r, uint32_t *first_row, uint32_t *num_rows)
{
    if (!r || !first_row || !num_rows) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    const ShardState &s = r->shard;
    if (s.world < 1) return fail(WS_ERR_INVALID_ARGUMENT, "renderer is not configured for sharding");
    const uint32_t y0 = s.band_y0[s.rank] * TILE, y1 = s.band_y0[s.rank + 1] * TILE;
    *first_row = y0 < s.height ? y0 : s.height;
    *num_rows = (y1 < s.height ? y1 : s.height) - *first_row;
    return WS_OK;
}

static size_t bytes_per_pixel(ws_format f) { return f == WS_FORMAT_RGBA8_UNORM ? 4 : (f == WS_FORMAT_RGBA16_FLOAT ? 8 : 16); }

extern "C" ws_status ws_renderer_render(ws_renderer *r, ws_pointcloud *pc, void *dst, size_t row_pitch,
                                        const double clear[4], void *cuda_stream)
{
    if (r && r->shard.world > 1) return fail(WS_ERR_INVALID_ARGUMENT, "sharded renderer: use ws_renderer_render_band");
    if (r && r->batch) return fail(WS_ERR_INVALID_ARGUMENT, "the prepared frame is a batch of views: use ws_renderer_render_views");
    return render_rows(r, pc, dst, row_pitch, clear, cuda_stream, 0, r ? r->h_uniforms.tiles_y : 0);
}

// the rows of this rank's band only; dst row 0 = first pixel row of the band (ws_renderer_shard_band)
extern "C" ws_status ws_renderer_render_band(ws_renderer *r, ws_pointcloud *pc, void *dst, size_t row_pitch,
                                             const double clear[4], void *cuda_stream)
{
    if (!r || r->shard.world < 1) return fail(WS_ERR_INVALID_ARGUMENT, "renderer is not configured for sharding");
    const ShardState &s = r->shard;
    return render_rows(r, pc, dst, row_pitch, clear, cuda_stream, s.band_y0[s.rank], s.band_y0[s.rank + 1] - s.band_y0[s.rank]);
}

// stage 3 for this rank's band, stored straight into the ROOT rank's assembled frame through the
// peer mapping (the gather of the bands is fused into the compositor's epilogue; the host layer only
// adds a barrier).  ws_renderer_shard_frame / _download read the assembled frame on the root.
extern "C" ws_status ws_renderer_render_band_to_root(ws_renderer *r, ws_pointcloud *pc, uint32_t root, const double clear[4], void *cuda_stream)
{
    if (!r || r->shard.world < 1 || root >= r->shard.world) return fail(WS_ERR_INVALID_ARGUMENT, "renderer is not configured for sharding / bad root");
    const ShardState &s = r->shard;
    if (!s.peer_frame[root][0]) return fail(WS_ERR_INVALID_ARGUMENT, "peer handles not imported");
    const size_t pitch = s.shard_frame_bytes / s.height;
    const uint32_t first = s.band_y0[s.rank] * TILE;
    if (first >= s.height) { r->rendered = true; return WS_OK; }
    return render_rows(r, pc, s.peer_frame[root][s.epoch & 1u] + (size_t)first * pitch, pitch, clear, cuda_stream, s.band_y0[s.rank], s.band_y0[s.rank + 1] - s.band_y0[s.rank]);
}
extern "C" ws_status ws_renderer_shard_frame(const ws_renderer *r, void **device_ptr, size_t *row_pitch_bytes)
{
    if (!r || !device_ptr || !row_pitch_bytes || r->shard.world < 1) return fail(WS_ERR_INVALID_ARGUMENT, "renderer is not configured for sharding");
    *device_ptr = r->shard.d_shard_frame[r->shard.epoch & 1u]; *row_pitch_bytes = r->shard.shard_frame_bytes / r->shard.height;
    return WS_OK;
}
extern "C" ws_status ws_renderer_shard_download(ws_renderer *r, void *dst_host, void *cuda_stream)
{
    if (!r || !dst_host || r->shard.world < 1) return fail(WS_ERR_INVALID_ARGUMENT, "renderer is not configured for sharding");
    CU(cudaSetDevice(r->ctx->device));
    CU(cudaMemcpyAsync(dst_host, r->shard.d_shard_frame[r->shard.epoch & 1u], r->shard.shard_frame_bytes, cudaMemcpyDeviceToHost, (cudaStream_t)cuda_stream));
    return WS_OK;
}

// stage 3 launch only (capturable): the compositor over tile rows [tile_y0, tile_y0 + tile_rows) into dst
static ws_status enqueue_composite(ws_renderer *r, void *dst, size_t row_pitch, const double clear[4], cudaStream_t stream,
                                   uint32_t tile_y0, uint32_t tile_rows, size_t view_stride)
{
    const FrameUniforms &U = r->h_uniforms;
    CompositeArgs a;
    memset(&a, 0, sizeof a);
    a.splats = r->d_splats; a.pair_slots = r->d_pslots[r->tile_out]; a.ranges = r->d_ranges;
    if (r->frame_split) {               // the far slab's list on top of the state the near slab left
        a.pair_slots = r->d_pslots[r->tile_out_far]; a.ranges = r->d_ranges + r->tiles_cap;
        a.mode = 2; a.state = r->d_state; a.tile_done = r->d_tile_done;
    }
    a.uniforms = r->d_uniforms; a.dst = dst; a.row_pitch = (uint32_t)row_pitch; a.format = (int)r->format;
    a.tile_y0 = tile_y0; a.active_cull = active_cull_default(); a.view_stride = view_stride;
    a.signal_flag = r->shard.pending_signal; a.signal_epoch = r->shard.d_epoch; a.done_counter = &r->d_counters->composite_done;
    r->shard.pending_signal = nullptr;
    for (int i = 0; i < 4; i++) a.clear[i] = clear ? (float)clear[i] : 0.f;
    if (r->timing) CU(cudaEventRecord(r->ev[EV_BLEND0], stream));
    if (tile_rows) CU(launch_composite(a, U.tiles_x, tile_rows, stream, r->views));
    if (r->timing) CU(cudaEventRecord(r->ev[EV_BLEND1], stream));
    return WS_OK;
}

// this frame's {V, P, pair_overflow, error_flags} -> a pinned slot; checked (never waited for) by later calls
static ws_status enqueue_status_copy(ws_renderer *r, cudaStream_t stream)
{
    const int slot = r->flag_next; r->flag_next = (slot + 1) % ws_renderer::FLAG_SLOTS;
    CU(cudaMemcpyAsync(r->h_flags + 4 * slot, r->d_counters, 16, cudaMemcpyDeviceToHost, stream));
    CU(cudaEventRecord(r->ev_flags[slot], stream));
    r->flags_pending[slot] = true;
    return WS_OK;
}

static ws_status render_rows(ws_renderer *r, ws_pointcloud *pc, void *dst, size_t row_pitch, const double clear[4],
                             void *cuda_stream, uint32_t tile_y0, uint32_t tile_rows, size_t view_stride)
{
    if (!r || !pc || !dst) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!r->prepared) return fail(WS_ERR_NOT_PREPARED, "prepare() must precede render()");
    const FrameUniforms &U = r->h_uniforms;
    const size_t bpp = bytes_per_pixel(r->format);
    if (row_pitch < (size_t)U.width * bpp || (row_pitch % bpp) != 0 || row_pitch > 0xffffffffu)
        return fail(WS_ERR_INVALID_ARGUMENT, "row_pitch_bytes too small or not a multiple of the pixel size");
    if (((uintptr_t)dst % bpp) != 0) return fail(WS_ERR_INVALID_ARGUMENT, "dst is not aligned to the pixel size");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(cudaSetDevice(r->ctx->device));
    ws_status st = enqueue_composite(r, dst, row_pitch, clear, stream, tile_y0, tile_rows, view_stride);
    if (st != WS_OK) return st;
    st = enqueue_status_copy(r, stream);
    if (st != WS_OK) return st;
    r->rendered = true;
    r->last_stream = stream;
    return WS_OK;
}

extern "C" ws_status ws_renderer_render_to_host(ws_renderer *r, ws_pointcloud *pc, void *dst_host, size_t row_pitch,
                                                const double clear[4], void *cuda_stream)
{
    if (!r || !pc || !dst_host) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!r->prepared) return fail(WS_ERR_NOT_PREPARED, "prepare() must precede render()");
    if (r->batch) return fail(WS_ERR_INVALID_ARGUMENT, "the prepared frame is a batch of views: use ws_renderer_render_views_to_host");
    const FrameUniforms &U = r->h_uniforms;
    const size_t bpp = bytes_per_pixel(r->format);
    const size_t tight = (size_t)U.width * bpp;
    if (row_pitch < tight) return fail(WS_ERR_INVALID_ARGUMENT, "row_pitch_bytes too small");
    const size_t need = tight * U.height;
    CU(cudaSetDevice(r->ctx->device));
    if (r->frame_bytes < need) {
        cudaFree(r->d_frame); r->d_frame = nullptr; r->frame_bytes = 0;
        CU(cudaMalloc(&r->d_frame, need));
        r->frame_bytes = need;
    }
    ws_status st = ws_renderer_render(r, pc, r->d_frame, tight, clear, cuda_stream);
    if (st != WS_OK) return st;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (row_pitch == tight) CU(cudaMemcpyAsync(dst_host, r->d_frame, need, cudaMemcpyDeviceToHost, stream));
    else CU(cudaMemcpy2DAsync(dst_host, row_pitch, r->d_frame, tight, tight, U.height, cudaMemcpyDeviceToHost, stream));
    return WS_OK;
}

static ws_status check_views_target(ws_renderer *r, ws_pointcloud *pc, const void *dst, size_t row_pitch, size_t view_stride)
{
    if (!r || !pc || !dst) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!r->prepared) return fail(WS_ERR_NOT_PREPARED, "prepare_views() must precede render_views()");
    if (!r->batch) return fail(WS_ERR_INVALID_ARGUMENT, "the prepared frame is a single view: use ws_renderer_render");
    if (r->shard.world > 0) return fail(WS_ERR_INVALID_ARGUMENT, "batches of views are not supported on a sharded renderer");
    const size_t bpp = bytes_per_pixel(r->format);
    if (view_stride < (size_t)r->h_uniforms.height * row_pitch || (view_stride % bpp) != 0)
        return fail(WS_ERR_INVALID_ARGUMENT, "view_stride_bytes smaller than height * row_pitch_bytes or not a multiple of the pixel size");
    return WS_OK;
}

extern "C" ws_status ws_renderer_render_views(ws_renderer *r, ws_pointcloud *pc, void *dst, size_t row_pitch,
                                              size_t view_stride, const double clear[4], void *cuda_stream)
{
    ws_status st = check_views_target(r, pc, dst, row_pitch, view_stride);
    if (st != WS_OK) return st;
    return render_rows(r, pc, dst, row_pitch, clear, cuda_stream, 0, r->h_uniforms.tiles_y / r->views, view_stride);
}

extern "C" ws_status ws_renderer_render_views_to_host(ws_renderer *r, ws_pointcloud *pc, void *dst_host, size_t row_pitch,
                                                      size_t view_stride, const double clear[4], void *cuda_stream)
{
    ws_status st = check_views_target(r, pc, dst_host, row_pitch, view_stride);
    if (st != WS_OK) return st;
    const FrameUniforms &U = r->h_uniforms;
    const size_t tight = (size_t)U.width * bytes_per_pixel(r->format);
    if (row_pitch < tight) return fail(WS_ERR_INVALID_ARGUMENT, "row_pitch_bytes too small");
    const size_t view_bytes = tight * U.height, need = view_bytes * r->views;
    CU(cudaSetDevice(r->ctx->device));
    if (r->frame_bytes < need) {
        cudaFree(r->d_frame); r->d_frame = nullptr; r->frame_bytes = 0;
        CU(cudaMalloc(&r->d_frame, need));
        r->frame_bytes = need;
    }
    st = ws_renderer_render_views(r, pc, r->d_frame, tight, view_bytes, clear, cuda_stream);
    if (st != WS_OK) return st;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (row_pitch == tight && view_stride == view_bytes) {
        CU(cudaMemcpyAsync(dst_host, r->d_frame, need, cudaMemcpyDeviceToHost, stream));
    } else {
        for (uint32_t v = 0; v < r->views; v++)
            CU(cudaMemcpy2DAsync(static_cast<uint8_t *>(dst_host) + v * view_stride, row_pitch, static_cast<uint8_t *>(r->d_frame) + v * view_bytes,
                                 tight, tight, U.height, cudaMemcpyDeviceToHost, stream));
    }
    return WS_OK;
}

extern "C" ws_status ws_renderer_views_num_visible_points(ws_renderer *r, uint32_t *out, uint32_t count)
{
    if (!r || !out) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!r->prepared) return fail(WS_ERR_NOT_PREPARED, "no frame prepared");
    if (!r->batch) return fail(WS_ERR_INVALID_ARGUMENT, "the prepared frame is not a batch of views");
    if (count < r->views) return fail(WS_ERR_INVALID_ARGUMENT, "count is smaller than the number of views");
    CU(cudaSetDevice(r->ctx->device));
    CU(cudaStreamSynchronize(r->last_stream));
    CU(cudaMemcpy(out, r->d_view_visible, r->views * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return WS_OK;
}

static ws_status read_counters(ws_renderer *r, FrameCounters *c)
{
    CU(cudaSetDevice(r->ctx->device));
    CU(cudaStreamSynchronize(r->last_stream));
    CU(cudaMemcpy(c, r->d_counters, sizeof *c, cudaMemcpyDeviceToHost));
    return WS_OK;
}

extern "C" ws_status ws_renderer_num_visible_points(ws_renderer *r, uint32_t *out)
{
    if (!r || !out) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!r->prepared) return fail(WS_ERR_NOT_PREPARED, "no frame prepared");
    FrameCounters c;
    ws_status st = read_counters(r, &c);
    if (st != WS_OK) return st;
    *out = c.num_visible;
    return WS_OK;
}

extern "C" ws_status ws_renderer_stats(ws_renderer *r, ws_frame_stats *s)
{
    if (!r || !s) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!r->prepared) return fail(WS_ERR_NOT_PREPARED, "no frame prepared");
    memset(s, 0, sizeof *s);
    FrameCounters c;
    ws_status st = read_counters(r, &c);
    if (st != WS_OK) return st;
    for (int i = 0; i < ws_renderer::FLAG_SLOTS; i++) r->flags_pending[i] = false;   // this call reports the frame's status itself
    const FrameUniforms &U = r->h_uniforms;
    s->num_points = r->last_n; s->num_visible = c.num_visible;
    s->num_pairs = (uint64_t)c.num_pairs + (r->frame_split ? c.num_pairs_near : 0u);      // split frames: near slab + what the far slab still had to emit
    s->pair_capacity = r->pair_cap; s->num_tiles = U.tiles_x * U.tiles_y; s->width = U.width; s->height = U.height;
    if (r->timing) {
        auto el = [&](int a, int b) { float ms = 0.f; return (cudaEventElapsedTime(&ms, r->ev[a], r->ev[b]) == cudaSuccess) ? ms : 0.f; };
        s->ms_preprocess = el(EV_START, EV_PRE);
        s->ms_depth_sort = el(EV_PRE, EV_DSORT);
        s->ms_binning = el(EV_DSORT, EV_BIN);
        s->ms_tile_sort = el(EV_BIN, EV_TSORT);
        s->ms_ranges = 0.f;                                   // fused into the last tile-sort pass
        if (r->rendered) s->ms_blend = el(EV_BLEND0, EV_BLEND1);
        if (r->frame_split) {                                 // near slab | near composite | far slab ... far composite
            s->ms_binning += el(EV_NEAR_BLEND, EV_BIN2);
            s->ms_tile_sort += el(EV_BIN2, EV_TSORT2);
            s->ms_blend += el(EV_TSORT, EV_NEAR_BLEND);
        }
        s->ms_sort = s->ms_depth_sort + s->ms_binning + s->ms_tile_sort;
        cudaGetLastError();
    }
    // a batch of K views (DESIGN.md "Batches of views"): V = sum of the V_v, T = K x tiles of one view, K x W x H pixels;
    // the cloud is read once and the SH of a Gaussian at most once (charged as min(V, N) at the batch's highest degree)
    const uint64_t N = r->last_n, V = c.num_visible;
    const uint64_t P = s->num_pairs < r->pair_cap ? s->num_pairs : r->pair_cap;
    const uint64_t T = s->num_tiles;
    const uint64_t px = (uint64_t)U.width * U.height * r->views;
    const uint64_t rec = r->compressed ? 24 : 28;
    const uint64_t ncoef = (uint64_t)(U.rs.max_sh_deg + 1) * (U.rs.max_sh_deg + 1);
    const uint64_t shb = r->compressed ? (12 + 3 * ncoef) : (U.rs.max_sh_deg >= 3 ? 96 : (U.rs.max_sh_deg == 2 ? 64 : 32));
    s->bytes_preprocess = N * 12 + N * rec + (V < N ? V : N) * shb + V * (20 + 4 + 4 + 8);   // count (xyz plane) + main
    s->bytes_sort = (uint64_t)r->depth_passes * V * 16 + V * 12 + P * 8 + (uint64_t)r->tile_passes * P * 16 + T * 8;
    s->bytes_blend = P * 24 + T * 8 + px * bytes_per_pixel(r->format);
    if (r->frame_split) {                                         // the far slab re-reads the slots + rectangles, the state goes out and in
        s->bytes_sort += (V - V / 4) * 12;
        s->bytes_blend += T * 8 + px * 32;
    }
    if (c.error_flags) return fail(WS_ERR_CUDA, (c.error_flags & 2u) ? "sharded frame: receive capacity exceeded" : ((c.error_flags & 4u) ? "sharded frame: a peer never arrived" : "internal: decoupled look-back watchdog fired"));
    if (c.pair_overflow) return fail(WS_ERR_PAIR_OVERFLOW, "pair capacity exceeded; raise it with ws_renderer_set_pair_capacity");
    return WS_OK;
}

extern "C" ws_status ws_renderer_read_buffer(ws_renderer *r, ws_buffer_id which, void *dst, size_t dst_bytes, size_t *written)
{
    if (!r || !dst) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!r->prepared) return fail(WS_ERR_NOT_PREPARED, "no frame prepared");
    if (r->batch) return fail(WS_ERR_UNSUPPORTED, "intermediate buffers of a batch of views cannot be read back");
    FrameCounters c;
    ws_status st = read_counters(r, &c);
    if (st != WS_OK) return st;
    const size_t V = c.num_visible;
    const size_t P = c.num_pairs < r->pair_cap ? c.num_pairs : r->pair_cap;
    const size_t T = (size_t)r->h_uniforms.tiles_x * r->h_uniforms.tiles_y;
    const void *src = nullptr; size_t bytes = 0;
    switch (which) {
    case WS_BUF_SPLATS_2D: src = r->d_splats; bytes = V * 20; break;
    case WS_BUF_DEPTH_KEYS:
        // slot-order keys live in keys[0] only until the first pass overwrote it on the way back;
        // with an even pass count keys[0] holds the SORTED keys, so slot order is re-derived below
        src = nullptr; bytes = V * 4; break;
    case WS_BUF_SORTED_INDICES: src = r->d_vals[r->depth_out]; bytes = V * 4; break;
    case WS_BUF_SORTED_KEYS: src = r->d_keys[r->depth_out]; bytes = V * 4; break;
    case WS_BUF_TILE_RECTS: src = r->d_rects; bytes = V * 8; break;
    // split frames: the pair buffers hold the far slab's list when the frame is over (c.num_pairs = its size)
    case WS_BUF_PAIR_TILES: src = r->d_ptiles[r->frame_split ? r->tile_out_far : r->tile_out]; bytes = P * 4; break;
    case WS_BUF_PAIR_SLOTS: src = r->d_pslots[r->frame_split ? r->tile_out_far : r->tile_out]; bytes = P * 4; break;
    case WS_BUF_TILE_RANGES: src = r->d_ranges + (r->frame_split ? r->tiles_cap : 0); bytes = T * 8; break;
    default: return fail(WS_ERR_INVALID_ARGUMENT, "unknown buffer id");
    }
    if (written) *written = bytes;
    if (dst_bytes < bytes) return fail(WS_ERR_INVALID_ARGUMENT, "destination too small");
    if (which == WS_BUF_DEPTH_KEYS) {
        // un-permute on the host: key_of_slot[sorted_idx[i]] = sorted_key[i]
        std::vector<uint32_t> sk(V), si(V);
        if (V) {
            CU(cudaMemcpy(sk.data(), r->d_keys[r->depth_out], V * 4, cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(si.data(), r->d_vals[r->depth_out], V * 4, cudaMemcpyDeviceToHost));
        }
        uint32_t *o = static_cast<uint32_t *>(dst);
        for (size_t i = 0; i < V; i++) if (si[i] < V) o[si[i]] = sk[i];
        return WS_OK;
    }
    if (which == WS_BUF_PAIR_TILES && sort_pass_can_skip_keys()) {
        // the last tile pass does not store the sorted tile ids (nothing on the frame path reads them);
        // the sorted list is "tile t repeated over [begin_t, end_t)", rebuilt here from the ranges
        std::vector<uint32_t> rg(2 * T);
        if (T) CU(cudaMemcpy(rg.data(), r->d_ranges + (r->frame_split ? r->tiles_cap : 0), T * 8, cudaMemcpyDeviceToHost));
        uint32_t *o = static_cast<uint32_t *>(dst);
        for (size_t i = 0; i < P; i++) o[i] = 0xffffffffu;
        for (size_t t = 0; t < T; t++) {
            const uint32_t b = rg[2 * t], e = ~rg[2 * t + 1];
            if (e > b) for (size_t i = b; i < e && i < P; i++) o[i] = (uint32_t)t;
        }
        return WS_OK;
    }
    if (bytes) CU(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    if (which == WS_BUF_TILE_RANGES) {      // device form is {begin, ~end} with 0xffffffff identities
        uint32_t *o = static_cast<uint32_t *>(dst);
        for (size_t t = 0; t < T; t++) {
            const uint32_t b = o[2 * t], e = ~o[2 * t + 1];
            if (e <= b) { o[2 * t] = 0; o[2 * t + 1] = 0; } else { o[2 * t + 1] = e; }
        }
    }
    return WS_OK;
}

extern "C" ws_status ws_renderer_camera_uniform(const ws_renderer *r, float out68[68])
{
    if (!r || !out68) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (r->batch) return fail(WS_ERR_UNSUPPORTED, "the prepared frame is a batch of views");
    memcpy(out68, &r->h_uniforms.cam, sizeof(CameraUniform));
    return WS_OK;
}
extern "C" ws_status ws_renderer_settings_uniform(const ws_renderer *r, void *out80)
{
    if (!r || !out80) return fail(WS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (r->batch) return fail(WS_ERR_UNSUPPORTED, "the prepared frame is a batch of views");
    memcpy(out80, &r->h_uniforms.rs, sizeof(RenderSettings));
    return WS_OK;
}

// ------------------------------------------------------------------------------------
// The sort on its own (GPURSSorter::record_sort, gpu_rs.rs:865-873; KAT gpu_rs.rs:295-331)
extern "C" ws_status ws_sort_pairs_u32(ws_context *ctx, uint32_t *keys, uint32_t *vals, uint32_t n, uint32_t key_bits, void *cuda_stream)
{
    if (!ctx) return fail(WS_ERR_INVALID_ARGUMENT, "NULL context");
    if (key_bits < 1 || key_bits > 32) return fail(WS_ERR_INVALID_ARGUMENT, "key_bits must be in [1,32]");
    if (n >= (1u << 30)) return fail(WS_ERR_UNSUPPORTED, "n must be < 2^30");
    if (n == 0) return WS_OK;
    if (!keys || !vals) return fail(WS_ERR_INVALID_ARGUMENT, "NULL buffer");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(cudaSetDevice(ctx->device));
    const int passes = (int)((key_bits + 7) / 8);
    const size_t sparts = ((size_t)n + SORT_PART - 1) / SORT_PART;
    // scratch: [n u32][tickets 4][hist 4*256][status passes*sparts*256] + ping-pong buffers
    const size_t gparts = (sparts + SORT_LB_GROUP - 1) / SORT_LB_GROUP;
    const size_t scratch_words = 8 + 4 * 256 + (size_t)passes * (sparts + gparts) * 256;
    uint32_t *scratch = nullptr, *k2 = nullptr, *v2 = nullptr;
    CU(cudaMalloc(&scratch, scratch_words * 4));
    cudaError_t e = cudaMalloc(&k2, (size_t)n * 4);
    if (e == cudaSuccess) e = cudaMalloc(&v2, (size_t)n * 4);
    if (e != cudaSuccess) { cudaFree(scratch); cudaFree(k2); cudaFree(v2); return fail_cuda(e, "cudaMalloc sort temp"); }
    ws_status st = WS_OK;
    do {
        e = cudaMemsetAsync(scratch, 0, scratch_words * 4, stream); if (e != cudaSuccess) break;
        e = cudaMemcpyAsync(scratch, &n, 4, cudaMemcpyHostToDevice, stream); if (e != cudaSuccess) break;
        uint32_t *n_ptr = scratch, *tickets = scratch + 4, *hist = scratch + 8, *status = scratch + 8 + 4 * 256;
        uint32_t *gstatus = status + (size_t)passes * sparts * 256;
        e = launch_sort_histogram(keys, n_ptr, n, hist, passes, ctx->sm_count * 4, stream); if (e != cudaSuccess) break;
        const int grid = ctx->sm_count * sort_pass_blocks_per_sm();
        uint32_t *kb[2] = {keys, k2}, *vb[2] = {vals, v2};
        int src = 0;
        for (int p = 0; p < passes && e == cudaSuccess; p++) {
            SortPassArgs a;
            a.keys_in = kb[src]; a.vals_in = vb[src]; a.keys_out = kb[src ^ 1]; a.vals_out = vb[src ^ 1];
            a.n_ptr = n_ptr; a.n_cap = n; a.status = status + (size_t)p * sparts * 256; a.ticket = tickets + p;
            a.hist = hist + p * 256; a.shift = 8u * (uint32_t)p; a.err = nullptr;
            a.gstatus = gstatus + (size_t)p * gparts * 256; a.ranges = nullptr;
            e = launch_sort_pass(a, grid, stream);
            src ^= 1;
        }
        if (e != cudaSuccess) break;
        if (src == 1) {   // odd pass count: bring the result home
            e = cudaMemcpyAsync(keys, k2, (size_t)n * 4, cudaMemcpyDeviceToDevice, stream); if (e != cudaSuccess) break;
            e = cudaMemcpyAsync(vals, v2, (size_t)n * 4, cudaMemcpyDeviceToDevice, stream); if (e != cudaSuccess) break;
        }
        e = cudaStreamSynchronize(stream);   // temp buffers are freed below
    } while (0);
    if (e != cudaSuccess) st = fail_cuda(e, "ws_sort_pairs_u32");
    cudaFree(scratch); cudaFree(k2); cudaFree(v2);
    return st;
}

extern "C" ws_status ws_sort_pairs_u32_host(ws_context *ctx, uint32_t *keys, uint32_t *vals, uint32_t n, uint32_t key_bits)
{
    if (!ctx) return fail(WS_ERR_INVALID_ARGUMENT, "NULL context");
    if (n == 0) return WS_OK;
    if (!keys || !vals) return fail(WS_ERR_INVALID_ARGUMENT, "NULL buffer");
    CU(cudaSetDevice(ctx->device));
    uint32_t *dk = nullptr, *dv = nullptr;
    CU(cudaMalloc(&dk, (size_t)n * 4));
    cudaError_t e = cudaMalloc(&dv, (size_t)n * 4);
    if (e != cudaSuccess) { cudaFree(dk); return fail_cuda(e, "cudaMalloc"); }
    ws_status st = WS_OK;
    e = cudaMemcpy(dk, keys, (size_t)n * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dv, vals, (size_t)n * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) st = fail_cuda(e, "cudaMemcpy H2D");
    if (st == WS_OK) st = ws_sort_pairs_u32(ctx, dk, dv, n, key_bits, nullptr);
    if (st == WS_OK) {
        e = cudaMemcpy(keys, dk, (size_t)n * 4, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(vals, dv, (size_t)n * 4, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) st = fail_cuda(e, "cudaMemcpy D2H");
    }
    cudaFree(dk); cudaFree(dv);
    return st;
}
