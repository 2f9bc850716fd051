/*
 * websplat_b200.h -- C ABI of the B200-native splat render path.
 *
 * This is the drop-in boundary for the ONE hot path of KeKsBoTer/web-splat:
 * GaussianRenderer::prepare + GaussianRenderer::render and the PointCloud GPU
 * layout they consume.  The reference exposes that path as a Rust struct API
 * (no FFI exists upstream); each entry point below names the reference item it
 * replaces (paths relative to the reference repo root).  INTEGRATION.md shows
 * the Rust `extern "C"` binding + safe wrapper that keeps the reference's names.
 *
 * Conventions
 *  - plain pointers and sizes only; opaque handles; no C++/torch/CUDA types.
 *    `cuda_stream` parameters are a `cudaStream_t` passed as `void*` (NULL =
 *    the legacy default stream).  This is the analogue of "records into the
 *    caller's CommandEncoder": all device work is enqueued on that stream and
 *    nothing blocks unless the call is documented as synchronising.
 *  - every function returns ws_status (0 = OK, negative = error); no exceptions
 *    or aborts cross the boundary (the reference unwrap()s / panics instead).
 *  - a ws_renderer is not re-entrant (same as `&mut self` in renderer.rs:191):
 *    one host thread per renderer handle, frames serialised by the caller.
 *  - there is no CPU fallback: every entry point that does work needs a CUDA
 *    device of compute capability 10.x and fails with WS_ERR_CUDA otherwise.
 */
#ifndef WEBSPLAT_B200_H
#define WEBSPLAT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define WS_API
#else
#define WS_API __attribute__((visibility("default")))
#endif

typedef int32_t ws_status;
enum {
    WS_OK = 0,
    WS_ERR_INVALID_ARGUMENT = -1,
    WS_ERR_CUDA = -2,            /* a CUDA runtime call failed / no usable device */
    WS_ERR_OUT_OF_MEMORY = -3,
    WS_ERR_PAIR_OVERFLOW = -4,   /* (tile, splat) pairs exceeded the pair capacity; frame incomplete */
    WS_ERR_NOT_PREPARED = -5,    /* render() without a preceding prepare() */
    WS_ERR_UNSUPPORTED = -6,
    WS_ERR_MISMATCH = -7         /* point cloud does not match the renderer's (sh_deg, compressed) */
};
WS_API const char *ws_status_string(ws_status s);
/* text of the last CUDA error seen by this thread's most recent failing call ("" if none) */
WS_API const char *ws_last_error(void);

typedef struct ws_context ws_context;       /* ~ WGPUContext (src/lib.rs:68-126): device + queue */
typedef struct ws_pointcloud ws_pointcloud; /* ~ PointCloud (src/pointcloud.rs:72-88) */
typedef struct ws_renderer ws_renderer;     /* ~ GaussianRenderer (src/renderer.rs:17-31) */

/* ---- context ---------------------------------------------------------------
 * replaces WGPUContext::new_instance (src/lib.rs:69-76): picks the device. */
WS_API ws_status ws_context_create(int cuda_device, ws_context **out);
WS_API void ws_context_destroy(ws_context *ctx);
WS_API int ws_context_device(const ws_context *ctx);
WS_API int ws_context_sm_count(const ws_context *ctx);

/* ---- value types -------------------------------------------------------- */
typedef struct { float min[3]; float max[3]; } ws_aabb;              /* Aabb<f32>, src/pointcloud.rs:398-403 */
typedef struct { int32_t zero_point; float scale; uint32_t _pad[2]; } ws_quantization;   /* src/pointcloud.rs:360-366 */
typedef struct { ws_quantization color_dc, color_rest, opacity, scaling_factor; } ws_quantization4; /* :389-396 */

/* GenericGaussianPointCloud (src/io/mod.rs:27-42): the CPU byte buffers in the
 * exact GPU layouts the reference uploads, plus metadata. */
typedef struct {
    const void *gaussians;      /* num_points x 28 B `Gaussian` (src/pointcloud.rs:38-45) or, compressed,
                                   num_points x 24 B `GaussianCompressed` (src/pointcloud.rs:14-24) */
    uint64_t num_points;
    const void *sh_coefs;       /* raw: num_points x 96 B [[f16;3];16] (src/io/mod.rs:65);
                                   compressed: i8, (sh_deg+1)^2*3 B per entry (src/io/npz.rs:183-196) */
    uint64_t sh_bytes;
    const void *covars;         /* compressed only: num_covars x 12 B `Covariance3D` (src/pointcloud.rs:63) */
    uint64_t num_covars;
    const ws_quantization4 *quantization;   /* compressed only */
    uint32_t sh_deg;
    uint32_t compressed;
    ws_aabb aabb;
    float center[3];
    int32_t has_up;  float up[3];
    int32_t has_mip_splatting; int32_t mip_splatting;
    int32_t has_kernel_size;   float kernel_size;
    int32_t has_background;    float background_color[3];
} ws_pointcloud_desc;

/* ---- PointCloud ------------------------------------------------------------
 * replaces PointCloud::new (src/pointcloud.rs:99-199).  Copies the host buffers to
 * HBM (synchronous); the caller keeps ownership of its memory. */
WS_API ws_status ws_pointcloud_create(ws_context *ctx, const ws_pointcloud_desc *desc, ws_pointcloud **out);
/* Compressed clouds (here and in ws_pointcloud_create_from_c3dgs): every record's geometry_idx / sh_idx is checked
 * once on the device against num_covars / the number of SH entries; an out-of-range index (wgpu would read zeros
 * through its bounds-checked storage buffers, a CUDA gather would fault) fails with WS_ERR_INVALID_ARGUMENT. */
/* .ply ingest: replaces PlyReader::new + read (src/io/ply.rs:28-48,165-195) and
 * GenericGaussianPointCloud::new (src/io/mod.rs:63-105).  `file_bytes` is the whole .ply file
 * (header + binary vertex block, little or big endian).  The header is parsed on the host; the
 * per-vertex conversion (sigmoid, exp, quaternion normalise, build_cov, f16, SH transpose),
 * the bounding box, centroid and plane normal run on the GPU.  sh_deg comes from the number of
 * f_* properties (io/ply.rs:102-114); `comment mip=`, `kernel_size=`, `background_color=` fill the
 * optional metadata (io/ply.rs:121-160).  ascii files -> WS_ERR_UNSUPPORTED like the reference's todo!(). */
/* Host-only header probe (no CUDA): what PlyReader::new extracts from the header (io/ply.rs:28-48),
 * with the same failure cases ws_pointcloud_create_from_ply reports. */
typedef struct {
    uint64_t num_points;       /* element vertex N, io/ply.rs:116-120 */
    uint64_t data_offset;      /* first byte after end_header */
    uint32_t sh_deg;           /* io/ply.rs:102-114 */
    uint32_t stride_bytes;     /* bytes per vertex */
    uint32_t big_endian;
    int32_t has_mip_splatting; int32_t mip_splatting;
    int32_t has_kernel_size;   float kernel_size;
    int32_t has_background;    float background_color[3];
} ws_ply_info;
WS_API ws_status ws_ply_probe(const void *file_bytes, uint64_t file_len, ws_ply_info *out);
WS_API ws_status ws_pointcloud_create_from_ply(ws_context *ctx, const void *file_bytes, uint64_t file_len, ws_pointcloud **out);
/* .npz (compressed 3DGS) ingest: replaces the array post-processing of NpzReader::read
 * (src/io/npz.rs:58-225) and GenericGaussianPointCloud::new_compressed (src/io/mod.rs:107-150).
 * The caller decodes the zip/npy container (the reference uses the npyz crate) and passes the arrays by
 * name as they are stored; the GPU assembles the 24-B GaussianCompressed records, interleaves the i8
 * SH codebook (dc then rest), dequantises rotation / scaling and builds the f16 covariance codebook
 * (build_cov, src/utils.rs:194-204), and reduces bbox (from the unit cube) / centroid / plane normal. */
typedef struct {
    const void *xyz;                 /* "xyz"              num_points x 3 f16 */
    const int8_t *opacity;           /* "opacity"          num_points i8 */
    const int8_t *scaling_factor;    /* "scaling_factor"   num_points i8, or NULL when the file has none */
    const int32_t *gaussian_indices; /* "gaussian_indices" num_points i32, or NULL (identity) */
    const int32_t *feature_indices;  /* "feature_indices"  num_points i32, or NULL (identity) */
    uint64_t num_points;
    const int8_t *scaling;           /* "scaling"          num_covars x 3 i8 */
    const int8_t *rotation;          /* "rotation"         num_covars x 4 i8 (w,x,y,z) */
    uint64_t num_covars;
    const int8_t *features_dc;       /* "features_dc"      num_features x 3 i8 */
    const int8_t *features_rest;     /* "features_rest"    num_features x ((sh_deg+1)^2 - 1) x 3 i8 */
    uint64_t num_features;
    uint32_t sh_deg;                 /* from features_rest.shape[1] + 1, src/io/npz.rs:33-37 */
    float scaling_scale;  int32_t scaling_zero_point;     /* src/io/npz.rs:65-68 */
    float rotation_scale; int32_t rotation_zero_point;    /* src/io/npz.rs:70-73 */
    ws_quantization4 quantization;   /* features_dc / features_rest / opacity / scaling_factor scale + zero point, src/io/npz.rs:216-221 */
    int32_t has_mip_splatting; int32_t mip_splatting;
    int32_t has_kernel_size;   float kernel_size;
    int32_t has_background;    float background_color[3];
} ws_c3dgs_arrays;
WS_API ws_status ws_pointcloud_create_from_c3dgs(ws_context *ctx, const ws_c3dgs_arrays *arrays, ws_pointcloud **out);
/* test / debug read-back of the resident layouts: which = 0 Gaussian records (28 B, or 24 B
 * compressed), 1 SH records (96 B raw; i8 codebook compressed), 2 xyz plane (12 B), 3 covariance
 * codebook (12 B, compressed only).  ws_pointcloud_buffer_bytes gives the size to allocate. */
WS_API uint64_t ws_pointcloud_buffer_bytes(const ws_pointcloud *pc, int32_t which);
WS_API ws_status ws_pointcloud_read(const ws_pointcloud *pc, int32_t which, void *dst, uint64_t dst_bytes);
WS_API void ws_pointcloud_destroy(ws_pointcloud *pc);
/* getters, src/pointcloud.rs:201-349 */
WS_API uint32_t ws_pointcloud_num_points(const ws_pointcloud *pc);
WS_API uint32_t ws_pointcloud_sh_deg(const ws_pointcloud *pc);
WS_API int32_t ws_pointcloud_compressed(const ws_pointcloud *pc);
WS_API ws_status ws_pointcloud_bbox(const ws_pointcloud *pc, ws_aabb *out);
WS_API ws_status ws_pointcloud_center(const ws_pointcloud *pc, float out[3]);
WS_API int32_t ws_pointcloud_up(const ws_pointcloud *pc, float out[3]);                 /* returns has_up */
WS_API int32_t ws_pointcloud_background_color(const ws_pointcloud *pc, float out[3]);   /* GenericGaussianPointCloud::background_color, src/io/mod.rs:41; returns 1 if Some */
WS_API int32_t ws_pointcloud_mip_splatting(const ws_pointcloud *pc, int32_t *out);      /* returns has_value */
WS_API int32_t ws_pointcloud_dilation_kernel_size(const ws_pointcloud *pc, float *out); /* returns has_value */

/* ---- camera helpers (host only, no device work) ----------------------------
 * Aabb::center / Aabb::radius (src/pointcloud.rs:441-448) and
 * PerspectiveCamera::fit_near_far (src/camera.rs:26-35). */
WS_API void ws_aabb_center(const ws_aabb *b, float out[3]);
WS_API float ws_aabb_radius(const ws_aabb *b);
WS_API void ws_camera_fit_near_far(const float position[3], const ws_aabb *aabb, float *znear, float *zfar);

/* ---- GaussianRenderer ---------------------------------------------------- */
typedef enum {            /* the three wgpu::TextureFormat values the reference's callers use */
    WS_FORMAT_RGBA8_UNORM = 0,   /* viewer default src/lib.rs:192-196, bin/measure.rs:184 */
    WS_FORMAT_RGBA16_FLOAT = 1,  /* --hdr, bin/render.rs:154 */
    WS_FORMAT_RGBA32_FLOAT = 2   /* bin/video.rs:186 */
} ws_format;

/* replaces GaussianRenderer::new (src/renderer.rs:33-123): specialised on
 * (format, sh_deg, compressed); serves any cloud with those properties. */
WS_API ws_status ws_renderer_create(ws_context *ctx, ws_format color_format, uint32_t sh_deg,
                                    int32_t compressed, ws_renderer **out);
WS_API void ws_renderer_destroy(ws_renderer *r);
WS_API ws_format ws_renderer_color_format(const ws_renderer *r);        /* src/renderer.rs:281-283 */

/* SplattingArgs (src/renderer.rs:587-599).  Option<T> fields become has_* flags. */
typedef struct {
    /* PerspectiveCamera (src/camera.rs:7-11) */
    float cam_position[3];
    float cam_rotation_wxyz[4];   /* cgmath Quaternion::new(w, xi, yj, zk); Matrix3::from(q) = world->camera */
    /* PerspectiveProjection (src/camera.rs:86-94); fov in radians */
    float fovx, fovy, znear, zfar, fov2view_ratio;
    uint32_t viewport[2];
    float gaussian_scaling;
    uint32_t max_sh_deg;
    int32_t has_mip_splatting; int32_t mip_splatting;
    int32_t has_kernel_size;   float kernel_size;
    int32_t has_clipping_box;  ws_aabb clipping_box;
    float walltime_secs;          /* Duration::as_secs_f32 (src/renderer.rs:643) */
    int32_t has_scene_center;  float scene_center[3];   /* ignored, as in the reference (src/renderer.rs:644) */
    int32_t has_scene_extend;  float scene_extend;
    double background_color[4];   /* wgpu::Color; not read by prepare (the caller clears with it) */
} ws_splatting_args;

/* replaces GaussianRenderer::prepare (src/renderer.rs:191-248): resolves the
 * uniforms (CameraUniform src/renderer.rs:321-343, SplattingArgsUniform
 * src/renderer.rs:620-651), (re)allocates the sort buffers when the point count
 * changed (src/renderer.rs:200-211) and enqueues stage 1 (preprocess) + stage 2
 * (sort; here: depth sort, tile binning, tile sort, tile ranges). Asynchronous. */
WS_API ws_status ws_renderer_prepare(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args,
                                     void *cuda_stream);
/* Frame status without synchronising: everything above is asynchronous, so a frame that turns out incomplete on the
 * device (pair capacity exceeded; internal error flags) cannot fail the call that enqueued it.  render() therefore
 * copies the frame's status words into pinned host memory behind the frame, and the NEXT prepare() (or sharded
 * frame call) that finds such a copy completed returns that earlier frame's error ONCE -- WS_ERR_PAIR_OVERFLOW or
 * WS_ERR_CUDA, with ws_last_error() saying "an earlier frame was incomplete" -- without enqueueing anything; calling
 * it again proceeds normally.  ws_renderer_stats() reports (and thereby consumes) the status of the frame it
 * synchronises.  A caller that needs the status of frame k before using its pixels calls ws_renderer_stats(). */

/* replaces GaussianRenderer::render (src/renderer.rs:250-260) together with the
 * caller's render pass (LoadOp::Clear(clear) on a target of color_format(),
 * src/lib.rs:451-462, bin/render.rs:108-123): enqueues stage 3 and writes the
 * finished frame to `dst_rgba` (DEVICE memory, row 0 = top row, `row_pitch_bytes`
 * >= width * bytes-per-pixel).  Must follow prepare on the same stream. Asynchronous. */
WS_API ws_status ws_renderer_render(ws_renderer *r, ws_pointcloud *pc, void *dst_rgba_device,
                                    size_t row_pitch_bytes, const double clear[4], void *cuda_stream);

/* render + download (bin/render.rs:187-246 download_texture): same as above into an
 * internal device frame, then an async device->host copy into `dst_rgba_host`
 * (pinned memory for a truly asynchronous copy).  Returns after enqueueing. */
WS_API ws_status ws_renderer_render_to_host(ws_renderer *r, ws_pointcloud *pc, void *dst_rgba_host,
                                            size_t row_pitch_bytes, const double clear[4], void *cuda_stream);

/* replaces GaussianRenderer::num_visible_points (src/renderer.rs:170-189). Synchronises the frame. */
WS_API ws_status ws_renderer_num_visible_points(ws_renderer *r, uint32_t *out);

/* The GPUStopwatch replacement (src/utils.rs:26-134; labels "preprocess", "sorting",
 * "rasterization": src/renderer.rs:220-239, src/lib.rs:447-467) plus counts.
 * Synchronises the last frame.  Returns WS_ERR_PAIR_OVERFLOW (with the stats still
 * filled in, num_pairs = pairs needed) when the frame overflowed the pair capacity. */
typedef struct {
    uint32_t num_points;      /* N */
    uint32_t num_visible;     /* V */
    uint64_t num_pairs;       /* P = sum over visible splats of 16x16 tiles touched */
    uint64_t pair_capacity;
    uint32_t num_tiles;       /* T */
    uint32_t width, height;
    float ms_preprocess;      /* stage 1 */
    float ms_sort;            /* stage 2: depth sort + tile binning + tile sort + ranges */
    float ms_blend;           /* stage 3 */
    float ms_depth_sort, ms_binning, ms_tile_sort, ms_ranges;   /* breakdown of ms_sort */
    uint64_t bytes_preprocess, bytes_sort, bytes_blend;         /* algorithmic HBM bytes (DESIGN.md) */
} ws_frame_stats;
WS_API ws_status ws_renderer_stats(ws_renderer *r, ws_frame_stats *out);

/* Capacity policy for the data-dependent pair list.  0 = automatic
 * (max(8*N, 1<<22)).  Takes effect at the next prepare(). */
WS_API ws_status ws_renderer_set_pair_capacity(ws_renderer *r, uint64_t max_pairs);
/* per-stage CUDA-event timing on/off (default on; costs 8 event records per frame) */
WS_API ws_status ws_renderer_set_timing(ws_renderer *r, int32_t enabled);
/* With timing off, prepare() replays one CUDA graph (2 clears + 14 kernels) per (cloud, viewport,
 * capacities) instead of 16 launches -- the frame-graph analogue of the reference recording one command
 * buffer per frame (src/lib.rs:415-500).  Default on; this switch exists for A/B measurements. */
WS_API ws_status ws_renderer_set_cuda_graphs(ws_renderer *r, int32_t enabled);
/* Occlusion split (single-GPU frames; enabled: 0 off, 1 on, negative = automatic, the default: on for clouds of at least
 * 2 M points, where the pairs it saves outweigh its six extra launches): the depth-sorted splats are binned, tile-sorted and composited
 * in two slabs, the nearest quarter first; a splat of the far slab whose tiles were all saturated by the near slab emits no
 * (tile, splat) pair.  Per pixel the blends and early-out tests are those of the one-pass frame: the image is
 * bit-identical, while num_pairs counts only the pairs that were emitted.  Turn it off to get the complete pair list
 * in the WS_BUF_PAIR_* / WS_BUF_TILE_RANGES read-backs (with the split they describe the far slab). */
WS_API ws_status ws_renderer_set_occlusion_split(ws_renderer *r, int32_t enabled);

/* ---- batches of views (new: the reference renders one view per prepare / render) --------------
 * K <= WS_MAX_VIEWS cameras of ONE cloud in one frame: stage 1 reads the cloud once for all views, stages 2-3 run
 * once over the K views stacked into one frame of K x tiles rows.  Every view is bit-identical to the same view
 * rendered alone through ws_renderer_prepare + ws_renderer_render.
 *  - args[0..num_views) must share the viewport; everything else (camera, clipping box, max_sh_deg, mip splatting,
 *    kernel size, gaussian_scaling, walltime) may differ.  Each view is checked like a single frame; in addition
 *    num_views of 0 or above WS_MAX_VIEWS, different viewports, a sharded renderer, render / render_to_host after
 *    prepare_views and render_views after prepare fail with WS_ERR_INVALID_ARGUMENT, and num_views x num_points
 *    >= 2^30 with WS_ERR_UNSUPPORTED.
 *  - after a batch, ws_renderer_read_buffer, ws_renderer_camera_uniform and ws_renderer_settings_uniform return
 *    WS_ERR_UNSUPPORTED.  ws_renderer_stats reports num_visible = sum of the per-view counts, num_pairs = the pairs of
 *    the batch, num_tiles = K x tiles, width / height of one view and the stage times of the whole batch;
 *    ws_renderer_num_visible_points returns the sum as well.
 *  - deferred frame status, the automatic pair capacity (K x max(8 N, 1<<22): what the views get one by one) and CUDA graphs (a graph of its own, so
 *    alternating single frames and batches does not recapture) work as for one frame.  The sort buffers are sized for
 *    K x N points: a renderer that alternates single frames and batches reallocates them at every switch; use one
 *    renderer per mode to avoid that. */
#define WS_MAX_VIEWS 8
/* stage 1 + 2 for num_views cameras of one cloud. Asynchronous. */
WS_API ws_status ws_renderer_prepare_views(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args,
                                           uint32_t num_views, void *cuda_stream);
/* stage 3 of the batch: view v lands at dst + v * view_stride_bytes (view_stride_bytes >= height * row_pitch_bytes,
 * a multiple of the pixel size). Asynchronous. */
WS_API ws_status ws_renderer_render_views(ws_renderer *r, ws_pointcloud *pc, void *dst_rgba_device, size_t row_pitch_bytes,
                                          size_t view_stride_bytes, const double clear[4], void *cuda_stream);
/* the same into an internal device buffer, then async copies to host memory (layout as above) */
WS_API ws_status ws_renderer_render_views_to_host(ws_renderer *r, ws_pointcloud *pc, void *dst_rgba_host, size_t row_pitch_bytes,
                                                  size_t view_stride_bytes, const double clear[4], void *cuda_stream);
/* per-view visible point counts V_v of the last batch into out[0..num_views) (count >= num_views). Synchronises. */
WS_API ws_status ws_renderer_views_num_visible_points(ws_renderer *r, uint32_t *out, uint32_t count);

/* ---- intermediate read-back (parity tests; synchronises) -------------------
 * Copies an intermediate buffer of the LAST prepared frame to host memory. */
typedef enum {
    WS_BUF_SPLATS_2D = 0,     /* V x 20 B `Splat` (src/pointcloud.rs:352-358), slot = Gaussian-index order */
    WS_BUF_DEPTH_KEYS = 1,    /* V x u32 sort_depths in slot order (preprocess.wgsl:273) */
    WS_BUF_SORTED_INDICES = 2,/* V x u32 payload after the depth sort = draw order (gaussian.wgsl:37) */
    WS_BUF_TILE_RECTS = 3,    /* V x 4 u16 {x0,y0,x1,y1} inclusive tile rect per slot (new design) */
    WS_BUF_PAIR_TILES = 4,    /* P x u32 tile id, sorted (new design) */
    WS_BUF_PAIR_SLOTS = 5,    /* P x u32 splat slot, sorted by (tile, depth key, slot) */
    WS_BUF_TILE_RANGES = 6,   /* T x {u32 begin, u32 end} into the pair list */
    WS_BUF_SORTED_KEYS = 7    /* V x u32 depth keys after the sort (ascending) */
} ws_buffer_id;
WS_API ws_status ws_renderer_read_buffer(ws_renderer *r, ws_buffer_id which, void *dst_host,
                                         size_t dst_bytes, size_t *bytes_written);

/* ---- the sort on its own ---------------------------------------------------
 * replaces GPURSSorter::record_sort (src/gpu_rs.rs:865-873) as used by the
 * reference's own self test GPURSSorter::test_sort (src/gpu_rs.rs:295-331):
 * stable ascending sort of n (u32 key, u32 payload) pairs in DEVICE memory,
 * in place (result lands back in keys/payload like the reference's ping-pong,
 * radix_sort.wgsl:482-509).  `key_bits` in [1,32]: only the low key_bits are
 * sorted (ceil(key_bits/8) onesweep passes). */
WS_API ws_status ws_sort_pairs_u32(ws_context *ctx, uint32_t *keys_device, uint32_t *payload_device,
                                   uint32_t n, uint32_t key_bits, void *cuda_stream);
/* host-memory convenience wrapper (uploads, sorts, downloads; synchronous) */
WS_API ws_status ws_sort_pairs_u32_host(ws_context *ctx, uint32_t *keys_host, uint32_t *payload_host,
                                        uint32_t n, uint32_t key_bits);

/* ---- sharded rendering over the GPUs of one box (new: the reference is single-GPU) -----------
 * One process per GPU.  Rank r uploads Gaussians [r*N/G, (r+1)*N/G) as its ws_pointcloud (with the
 * GLOBAL aabb/center metadata) and owns a band of 16-pixel tile rows of the frame.  Per frame:
 *   shard_begin     stage 1 on the local shard + routing counts; writes this rank's row of the
 *                   G x G count matrix (G u32, DEVICE memory) to totals_row_device
 *   [host layer]    all-gather the rows (NCCL), G*G u32 on every rank
 *   shard_exchange  one kernel that stores every visible splat (20-B Splat, key, clipped tile
 *                   rectangle) directly into the owning ranks' buffers through peer-mapped pointers
 *   [host layer]    cross-rank barrier (e.g. a 4-byte NCCL all-reduce on the same stream)
 *   shard_finish    depth sort, binning, tile sort on what this rank received
 *   render_band     stage 3 for the rank's rows; the host layer gathers the bands.
 * Records arrive in global Gaussian-index order, so the result is bit-identical to one GPU.
 * Setup: shard_configure on every rank, exchange the 6x64-byte handles of shard_export (e.g.
 * torch.distributed.all_gather), shard_import.  Buffers never move after configure. */
WS_API ws_status ws_renderer_shard_configure(ws_renderer *r, uint32_t rank, uint32_t world, uint64_t total_points,
                                             uint32_t local_points, uint32_t width, uint32_t height);
WS_API ws_status ws_renderer_shard_export(ws_renderer *r, void *handles_6x64);
WS_API ws_status ws_renderer_shard_import(ws_renderer *r, const void *all_handles_world_x_6x64);
WS_API ws_status ws_renderer_shard_begin(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args,
                                         uint32_t *totals_row_device, void *cuda_stream);
WS_API ws_status ws_renderer_shard_exchange(ws_renderer *r, const uint32_t *matrix_device, void *cuda_stream);
WS_API ws_status ws_renderer_shard_finish(ws_renderer *r, const uint32_t *matrix_device, void *cuda_stream);
WS_API ws_status ws_renderer_shard_band(const ws_renderer *r, uint32_t *first_row, uint32_t *num_rows);
WS_API ws_status ws_renderer_render_band(ws_renderer *r, ws_pointcloud *pc, void *dst_rgba_device, size_t row_pitch_bytes,
                                         const double clear[4], void *cuda_stream);
/* stage 3 with the band gather fused in: the band's pixels are stored directly into the ROOT
 * rank's assembled frame (peer memory); after a cross-rank barrier the root reads it with
 * ws_renderer_shard_frame (device pointer) or ws_renderer_shard_download (async copy to host). */
WS_API ws_status ws_renderer_render_band_to_root(ws_renderer *r, ws_pointcloud *pc, uint32_t root, const double clear[4], void *cuda_stream);
WS_API ws_status ws_renderer_shard_frame(const ws_renderer *r, void **device_ptr, size_t *row_pitch_bytes);
/* The same frame (begin, count rows, exchange, barrier, finish, band -> root, "all bands landed") in ONE
 * call and WITHOUT any host-side collective: the count rows, the barrier and the band-arrival signal are
 * epoch flags the kernels write into the peers' mailboxes (release/acquire at system scope over NVLink).
 * Every rank calls it once per frame; the assembled frame is in rank `root`'s frame buffer.  The root keeps
 * TWO frame buffers (frame parity), so frame f can be downloaded on another stream while frame f+1 is
 * produced; the root must not start frame f+2 before that download has finished (stream/event ordering). */
WS_API ws_status ws_renderer_shard_frame_to_root(ws_renderer *r, ws_pointcloud *pc, const ws_splatting_args *args,
                                                 uint32_t root, const double clear[4], void *cuda_stream);
/* Cost-balanced bands: replace the equal tile-row split of ws_renderer_shard_configure.  band_y0 has world + 1
 * entries, 0 = band_y0[0] < ... < band_y0[world] = ceil(height / 16); rank d owns tile rows
 * [band_y0[d], band_y0[d+1]).  Every rank must pass the same array, between frames. */
WS_API ws_status ws_renderer_shard_set_bands(ws_renderer *r, const uint32_t *band_y0, uint32_t count);
WS_API ws_status ws_renderer_shard_get_bands(const ws_renderer *r, uint32_t *band_y0, uint32_t count);
/* Several sharded frames in flight per GPU (one renderer + one stream per frame slot): the peer-flag waits of
 * ws_renderer_shard_frame_to_root move into one-warp gate kernels so that no wide kernel ever spins. */
WS_API ws_status ws_renderer_shard_set_gated(ws_renderer *r, int32_t enabled);
WS_API ws_status ws_renderer_shard_download(ws_renderer *r, void *dst_rgba_host, void *cuda_stream);

/* ---- uniforms, for inspection (renderer.rs:125, 285) ------------------------
 * CameraUniform (272 B, src/renderer.rs:290-306) and SplattingArgsUniform
 * (80 B, src/renderer.rs:604-619) exactly as the reference would upload them. */
WS_API ws_status ws_renderer_camera_uniform(const ws_renderer *r, float out68[68]);
WS_API ws_status ws_renderer_settings_uniform(const ws_renderer *r, void *out80);

WS_API const char *ws_version(void);

#ifdef __cplusplus
}
#endif
#endif /* WEBSPLAT_B200_H */
