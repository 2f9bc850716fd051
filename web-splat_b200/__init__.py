"""websplat_b200 -- Python host layer over the C ABI (include/websplat_b200.h).

The reference's render API is a Rust struct API (src/renderer.rs, src/pointcloud.rs,
src/camera.rs).  No Rust toolchain exists in this image, so the host side above the
C ABI is mirrored here with the SAME names, argument meaning and error behaviour:

    reference (Rust)                                   here
    -------------------------------------------------  -----------------------------------
    WGPUContext::new_instance      lib.rs:69-76        Context(device)
    GenericGaussianPointCloud      io/mod.rs:27-42     GenericGaussianPointCloud
    PointCloud::new(device, pc)    pointcloud.rs:99    PointCloud.new(ctx, pc)
    Aabb<f32>                      pointcloud.rs:398   Aabb
    PerspectiveCamera / Projection camera.rs:7-11,86   PerspectiveCamera / PerspectiveProjection
    SplattingArgs                  renderer.rs:587     SplattingArgs
    GaussianRenderer::new          renderer.rs:33      GaussianRenderer.new(ctx, fmt, sh_deg, compressed)
    GaussianRenderer::prepare      renderer.rs:191     GaussianRenderer.prepare(stream, pc, args)
    GaussianRenderer::render       renderer.rs:250     GaussianRenderer.render(target, pc, clear, stream)
    (new: K views of one cloud)                        GaussianRenderer.prepare_views / render_views
    num_visible_points             renderer.rs:170     GaussianRenderer.num_visible_points()
    GPUStopwatch                   utils.rs:26-134     GaussianRenderer.stats()

This module is plumbing only: every frame is produced by the hand-written sm_100a kernels in
csrc/ through libwebsplat_b200.so.  There is NO CPU fallback: if the library is missing it
is built with nvcc; if no CUDA device is present Context() raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libwebsplat_b200.so")

WS_OK = 0
WS_ERR_INVALID_ARGUMENT = -1
WS_ERR_CUDA = -2
WS_ERR_OUT_OF_MEMORY = -3
WS_ERR_PAIR_OVERFLOW = -4
WS_ERR_NOT_PREPARED = -5
WS_ERR_UNSUPPORTED = -6
WS_ERR_MISMATCH = -7

FORMAT_RGBA8_UNORM = 0     # wgpu::TextureFormat::Rgba8Unorm
FORMAT_RGBA16_FLOAT = 1    # Rgba16Float
FORMAT_RGBA32_FLOAT = 2    # Rgba32Float
_BPP = {0: 4, 1: 8, 2: 16}
_NP_PIXEL = {0: (np.uint8, 4), 1: (np.float16, 4), 2: (np.float32, 4)}

BUF_SPLATS_2D, BUF_DEPTH_KEYS, BUF_SORTED_INDICES, BUF_TILE_RECTS = 0, 1, 2, 3
BUF_PAIR_TILES, BUF_PAIR_SLOTS, BUF_TILE_RANGES, BUF_SORTED_KEYS = 4, 5, 6, 7


class WsError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("websplat_b200: %s (status %d)%s" % (_status_string(status), status, (": " + msg) if msg else ""))
        self.status = status


# ---- ctypes mirror of the header ---------------------------------------------------------
class ws_aabb(C.Structure):
    _fields_ = [("min", C.c_float * 3), ("max", C.c_float * 3)]


class ws_quantization(C.Structure):
    _fields_ = [("zero_point", C.c_int32), ("scale", C.c_float), ("_pad", C.c_uint32 * 2)]


class ws_quantization4(C.Structure):
    _fields_ = [("color_dc", ws_quantization), ("color_rest", ws_quantization),
                ("opacity", ws_quantization), ("scaling_factor", ws_quantization)]


class ws_pointcloud_desc(C.Structure):
    _fields_ = [
        ("gaussians", C.c_void_p), ("num_points", C.c_uint64),
        ("sh_coefs", C.c_void_p), ("sh_bytes", C.c_uint64),
        ("covars", C.c_void_p), ("num_covars", C.c_uint64),
        ("quantization", C.POINTER(ws_quantization4)),
        ("sh_deg", C.c_uint32), ("compressed", C.c_uint32),
        ("aabb", ws_aabb), ("center", C.c_float * 3),
        ("has_up", C.c_int32), ("up", C.c_float * 3),
        ("has_mip_splatting", C.c_int32), ("mip_splatting", C.c_int32),
        ("has_kernel_size", C.c_int32), ("kernel_size", C.c_float),
        ("has_background", C.c_int32), ("background_color", C.c_float * 3),
    ]


class ws_c3dgs_arrays(C.Structure):
    _fields_ = [("xyz", C.c_void_p), ("opacity", C.c_void_p), ("scaling_factor", C.c_void_p), ("gaussian_indices", C.c_void_p),
                ("feature_indices", C.c_void_p), ("num_points", C.c_uint64), ("scaling", C.c_void_p), ("rotation", C.c_void_p),
                ("num_covars", C.c_uint64), ("features_dc", C.c_void_p), ("features_rest", C.c_void_p), ("num_features", C.c_uint64),
                ("sh_deg", C.c_uint32), ("scaling_scale", C.c_float), ("scaling_zero_point", C.c_int32),
                ("rotation_scale", C.c_float), ("rotation_zero_point", C.c_int32), ("quantization", ws_quantization4),
                ("has_mip_splatting", C.c_int32), ("mip_splatting", C.c_int32), ("has_kernel_size", C.c_int32),
                ("kernel_size", C.c_float), ("has_background", C.c_int32), ("background_color", C.c_float * 3)]


class ws_ply_info(C.Structure):
    _fields_ = [("num_points", C.c_uint64), ("data_offset", C.c_uint64), ("sh_deg", C.c_uint32), ("stride_bytes", C.c_uint32),
                ("big_endian", C.c_uint32), ("has_mip_splatting", C.c_int32), ("mip_splatting", C.c_int32),
                ("has_kernel_size", C.c_int32), ("kernel_size", C.c_float), ("has_background", C.c_int32),
                ("background_color", C.c_float * 3)]


class ws_splatting_args(C.Structure):
    _fields_ = [
        ("cam_position", C.c_float * 3), ("cam_rotation_wxyz", C.c_float * 4),
        ("fovx", C.c_float), ("fovy", C.c_float), ("znear", C.c_float), ("zfar", C.c_float),
        ("fov2view_ratio", C.c_float),
        ("viewport", C.c_uint32 * 2), ("gaussian_scaling", C.c_float), ("max_sh_deg", C.c_uint32),
        ("has_mip_splatting", C.c_int32), ("mip_splatting", C.c_int32),
        ("has_kernel_size", C.c_int32), ("kernel_size", C.c_float),
        ("has_clipping_box", C.c_int32), ("clipping_box", ws_aabb),
        ("walltime_secs", C.c_float),
        ("has_scene_center", C.c_int32), ("scene_center", C.c_float * 3),
        ("has_scene_extend", C.c_int32), ("scene_extend", C.c_float),
        ("background_color", C.c_double * 4),
    ]


class ws_frame_stats(C.Structure):
    _fields_ = [
        ("num_points", C.c_uint32), ("num_visible", C.c_uint32), ("num_pairs", C.c_uint64),
        ("pair_capacity", C.c_uint64), ("num_tiles", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32),
        ("ms_preprocess", C.c_float), ("ms_sort", C.c_float), ("ms_blend", C.c_float),
        ("ms_depth_sort", C.c_float), ("ms_binning", C.c_float), ("ms_tile_sort", C.c_float), ("ms_ranges", C.c_float),
        ("bytes_preprocess", C.c_uint64), ("bytes_sort", C.c_uint64), ("bytes_blend", C.c_uint64),
    ]


# every symbol include/websplat_b200.h declares (tests check the .so exports all of them)
EXPORTED_SYMBOLS = [
    "ws_status_string", "ws_last_error", "ws_context_create", "ws_context_destroy", "ws_context_device",
    "ws_context_sm_count", "ws_pointcloud_create", "ws_pointcloud_create_from_ply", "ws_pointcloud_create_from_c3dgs", "ws_pointcloud_read",
    "ws_pointcloud_buffer_bytes", "ws_ply_probe",
    "ws_pointcloud_background_color", "ws_pointcloud_destroy", "ws_pointcloud_num_points",
    "ws_pointcloud_sh_deg", "ws_pointcloud_compressed", "ws_pointcloud_bbox", "ws_pointcloud_center",
    "ws_pointcloud_up", "ws_pointcloud_mip_splatting", "ws_pointcloud_dilation_kernel_size",
    "ws_aabb_center", "ws_aabb_radius", "ws_camera_fit_near_far", "ws_renderer_create", "ws_renderer_destroy",
    "ws_renderer_color_format", "ws_renderer_prepare", "ws_renderer_render", "ws_renderer_render_to_host",
    "ws_renderer_num_visible_points", "ws_renderer_stats", "ws_renderer_set_pair_capacity",
    "ws_renderer_set_timing", "ws_renderer_set_cuda_graphs", "ws_renderer_set_occlusion_split", "ws_renderer_read_buffer", "ws_sort_pairs_u32", "ws_sort_pairs_u32_host",
    "ws_renderer_camera_uniform", "ws_renderer_settings_uniform", "ws_version",
    "ws_renderer_shard_configure", "ws_renderer_shard_export", "ws_renderer_shard_import", "ws_renderer_shard_begin",
    "ws_renderer_shard_exchange", "ws_renderer_shard_finish", "ws_renderer_shard_band", "ws_renderer_render_band",
    "ws_renderer_render_band_to_root", "ws_renderer_shard_frame", "ws_renderer_shard_download",
    "ws_renderer_shard_frame_to_root", "ws_renderer_shard_set_bands", "ws_renderer_shard_get_bands", "ws_renderer_shard_set_gated",
    "ws_renderer_prepare_views", "ws_renderer_render_views", "ws_renderer_render_views_to_host", "ws_renderer_views_num_visible_points",
]

MAX_VIEWS = 8              # WS_MAX_VIEWS: views per batch

_lib = None


def build_library(force=False):
    """Compile libwebsplat_b200.so in-tree with nvcc (sm_100a).  No fallback if nvcc fails."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ws_build", os.path.join(_HERE, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build(force=force)[0]


def lib():
    """Load (building if necessary) the CUDA library.  Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        build_library()
    L = C.CDLL(LIB_PATH)
    vp, u32, i32, u64, f32 = C.c_void_p, C.c_uint32, C.c_int32, C.c_uint64, C.c_float
    sig = {
        "ws_status_string": (C.c_char_p, [i32]),
        "ws_last_error": (C.c_char_p, []),
        "ws_version": (C.c_char_p, []),
        "ws_context_create": (i32, [C.c_int, C.POINTER(vp)]),
        "ws_context_destroy": (None, [vp]),
        "ws_context_device": (C.c_int, [vp]),
        "ws_context_sm_count": (C.c_int, [vp]),
        "ws_pointcloud_create": (i32, [vp, C.POINTER(ws_pointcloud_desc), C.POINTER(vp)]),
        "ws_pointcloud_create_from_ply": (i32, [vp, vp, u64, C.POINTER(vp)]),
        "ws_pointcloud_create_from_c3dgs": (i32, [vp, C.POINTER(ws_c3dgs_arrays), C.POINTER(vp)]),
        "ws_pointcloud_buffer_bytes": (u64, [vp, i32]),
        "ws_pointcloud_read": (i32, [vp, i32, vp, u64]),
        "ws_ply_probe": (i32, [vp, u64, C.POINTER(ws_ply_info)]),
        "ws_pointcloud_destroy": (None, [vp]),
        "ws_pointcloud_num_points": (u32, [vp]),
        "ws_pointcloud_sh_deg": (u32, [vp]),
        "ws_pointcloud_compressed": (i32, [vp]),
        "ws_pointcloud_bbox": (i32, [vp, C.POINTER(ws_aabb)]),
        "ws_pointcloud_center": (i32, [vp, C.POINTER(f32 * 3)]),
        "ws_pointcloud_up": (i32, [vp, C.POINTER(f32 * 3)]),
        "ws_pointcloud_background_color": (i32, [vp, C.POINTER(f32 * 3)]),
        "ws_pointcloud_mip_splatting": (i32, [vp, C.POINTER(i32)]),
        "ws_pointcloud_dilation_kernel_size": (i32, [vp, C.POINTER(f32)]),
        "ws_aabb_center": (None, [C.POINTER(ws_aabb), C.POINTER(f32 * 3)]),
        "ws_aabb_radius": (f32, [C.POINTER(ws_aabb)]),
        "ws_camera_fit_near_far": (None, [C.POINTER(f32 * 3), C.POINTER(ws_aabb), C.POINTER(f32), C.POINTER(f32)]),
        "ws_renderer_create": (i32, [vp, C.c_int, u32, i32, C.POINTER(vp)]),
        "ws_renderer_destroy": (None, [vp]),
        "ws_renderer_color_format": (C.c_int, [vp]),
        "ws_renderer_prepare": (i32, [vp, vp, C.POINTER(ws_splatting_args), vp]),
        "ws_renderer_render": (i32, [vp, vp, vp, C.c_size_t, C.POINTER(C.c_double * 4), vp]),
        "ws_renderer_render_to_host": (i32, [vp, vp, vp, C.c_size_t, C.POINTER(C.c_double * 4), vp]),
        "ws_renderer_num_visible_points": (i32, [vp, C.POINTER(u32)]),
        "ws_renderer_stats": (i32, [vp, C.POINTER(ws_frame_stats)]),
        "ws_renderer_set_pair_capacity": (i32, [vp, u64]),
        "ws_renderer_set_timing": (i32, [vp, i32]),
        "ws_renderer_set_cuda_graphs": (i32, [vp, i32]),
        "ws_renderer_set_occlusion_split": (i32, [vp, i32]),
        "ws_renderer_read_buffer": (i32, [vp, C.c_int, vp, C.c_size_t, C.POINTER(C.c_size_t)]),
        "ws_sort_pairs_u32": (i32, [vp, vp, vp, u32, u32, vp]),
        "ws_sort_pairs_u32_host": (i32, [vp, vp, vp, u32, u32]),
        "ws_renderer_camera_uniform": (i32, [vp, C.POINTER(f32 * 68)]),
        "ws_renderer_settings_uniform": (i32, [vp, vp]),
        "ws_renderer_shard_configure": (i32, [vp, u32, u32, u64, u32, u32, u32]),
        "ws_renderer_shard_export": (i32, [vp, vp]),
        "ws_renderer_shard_import": (i32, [vp, vp]),
        "ws_renderer_shard_begin": (i32, [vp, vp, C.POINTER(ws_splatting_args), vp, vp]),
        "ws_renderer_shard_exchange": (i32, [vp, vp, vp]),
        "ws_renderer_shard_finish": (i32, [vp, vp, vp]),
        "ws_renderer_shard_band": (i32, [vp, C.POINTER(u32), C.POINTER(u32)]),
        "ws_renderer_render_band": (i32, [vp, vp, vp, C.c_size_t, C.POINTER(C.c_double * 4), vp]),
        "ws_renderer_render_band_to_root": (i32, [vp, vp, u32, C.POINTER(C.c_double * 4), vp]),
        "ws_renderer_shard_frame": (i32, [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]),
        "ws_renderer_shard_download": (i32, [vp, vp, vp]),
        "ws_renderer_shard_set_bands": (i32, [vp, C.POINTER(u32), u32]),
        "ws_renderer_shard_get_bands": (i32, [vp, C.POINTER(u32), u32]),
        "ws_renderer_shard_set_gated": (i32, [vp, i32]),
        "ws_renderer_shard_frame_to_root": (i32, [vp, vp, C.POINTER(ws_splatting_args), u32, C.POINTER(C.c_double * 4), vp]),
        "ws_renderer_prepare_views": (i32, [vp, vp, C.POINTER(ws_splatting_args), u32, vp]),
        "ws_renderer_render_views": (i32, [vp, vp, vp, C.c_size_t, C.c_size_t, C.POINTER(C.c_double * 4), vp]),
        "ws_renderer_render_views_to_host": (i32, [vp, vp, vp, C.c_size_t, C.c_size_t, C.POINTER(C.c_double * 4), vp]),
        "ws_renderer_views_num_visible_points": (i32, [vp, C.POINTER(u32), u32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _status_string(s):
    try:
        return lib().ws_status_string(s).decode()
    except Exception:
        return "status"


def _check(status):
    if status != WS_OK:
        raise WsError(status, lib().ws_last_error().decode())


def _f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


# ---- value types -----------------------------------------------------------------------------
class Aabb:
    """Aabb<f32>, pointcloud.rs:398-463."""

    def __init__(self, min, max):
        self.min = np.asarray(min, dtype=np.float32).reshape(3)
        self.max = np.asarray(max, dtype=np.float32).reshape(3)

    def _c(self):
        return ws_aabb(_f3(self.min), _f3(self.max))

    def center(self):
        out = (C.c_float * 3)()
        lib().ws_aabb_center(C.byref(self._c()), C.byref(out))
        return np.array(out[:], dtype=np.float32)

    def radius(self):
        return float(lib().ws_aabb_radius(C.byref(self._c())))


class PerspectiveProjection:
    """camera.rs:86-94; fov in radians."""

    def __init__(self, fovx, fovy, znear, zfar, fov2view_ratio=1.0):
        self.fovx, self.fovy = float(fovx), float(fovy)
        self.znear, self.zfar = float(znear), float(zfar)
        self.fov2view_ratio = float(fov2view_ratio)


class PerspectiveCamera:
    """camera.rs:7-11.  rotation = (w, x, y, z); Matrix3::from(rotation) is world->camera."""

    def __init__(self, position, rotation, projection):
        self.position = np.asarray(position, dtype=np.float32).reshape(3)
        self.rotation = np.asarray(rotation, dtype=np.float32).reshape(4)
        self.projection = projection

    def fit_near_far(self, aabb):
        """camera.rs:26-35."""
        zn, zf = C.c_float(), C.c_float()
        lib().ws_camera_fit_near_far(C.byref(_f3(self.position)), C.byref(aabb._c()), C.byref(zn), C.byref(zf))
        self.projection.znear, self.projection.zfar = zn.value, zf.value


class SplattingArgs:
    """renderer.rs:587-599 (None = the Rust Option::None)."""

    def __init__(self, camera, viewport, gaussian_scaling=1.0, max_sh_deg=3, mip_splatting=None,
                 kernel_size=None, clipping_box=None, walltime=100.0, scene_center=None,
                 scene_extend=None, background_color=(0.0, 0.0, 0.0, 0.0)):
        self.camera = camera
        self.viewport = (int(viewport[0]), int(viewport[1]))
        self.gaussian_scaling = float(gaussian_scaling)
        self.max_sh_deg = int(max_sh_deg)
        self.mip_splatting = mip_splatting
        self.kernel_size = kernel_size
        self.clipping_box = clipping_box
        self.walltime = float(walltime)
        self.scene_center = scene_center
        self.scene_extend = scene_extend
        self.background_color = tuple(float(c) for c in background_color)

    def _c(self):
        a = ws_splatting_args()
        cam = self.camera
        a.cam_position = _f3(cam.position)
        a.cam_rotation_wxyz = (C.c_float * 4)(*[float(x) for x in cam.rotation])
        p = cam.projection
        a.fovx, a.fovy, a.znear, a.zfar, a.fov2view_ratio = p.fovx, p.fovy, p.znear, p.zfar, p.fov2view_ratio
        a.viewport = (C.c_uint32 * 2)(*self.viewport)
        a.gaussian_scaling = self.gaussian_scaling
        a.max_sh_deg = self.max_sh_deg
        a.has_mip_splatting = self.mip_splatting is not None
        a.mip_splatting = bool(self.mip_splatting)
        a.has_kernel_size = self.kernel_size is not None
        a.kernel_size = float(self.kernel_size or 0.0)
        a.has_clipping_box = self.clipping_box is not None
        if self.clipping_box is not None:
            a.clipping_box = self.clipping_box._c()
        a.walltime_secs = self.walltime
        a.has_scene_center = self.scene_center is not None
        if self.scene_center is not None:
            a.scene_center = _f3(self.scene_center)
        a.has_scene_extend = self.scene_extend is not None
        a.scene_extend = float(self.scene_extend or 0.0)
        a.background_color = (C.c_double * 4)(*self.background_color)
        return a


class GenericGaussianPointCloud:
    """io/mod.rs:27-42: host byte buffers in the GPU layouts + metadata."""

    def __init__(self, gaussians, sh_coefs, sh_deg, num_points, aabb, center, compressed=False, covars=None,
                 quantization=None, kernel_size=None, mip_splatting=None, background_color=None, up=None):
        self.gaussians = np.ascontiguousarray(gaussians).view(np.uint8).reshape(-1)
        self.sh_coefs = np.ascontiguousarray(sh_coefs).view(np.uint8).reshape(-1)
        self.sh_deg = int(sh_deg)
        self.num_points = int(num_points)
        self.aabb = aabb
        self.center = np.asarray(center, dtype=np.float32).reshape(3)
        self.compressed = bool(compressed)
        self.covars = None if covars is None else np.ascontiguousarray(covars).view(np.uint8).reshape(-1)
        self.quantization = quantization      # dict name -> (zero_point, scale)
        self.kernel_size, self.mip_splatting = kernel_size, mip_splatting
        self.background_color, self.up = background_color, up

    def quantization_struct(self):
        q = ws_quantization4()
        if self.quantization:
            for name in ("color_dc", "color_rest", "opacity", "scaling_factor"):
                zp, sc = self.quantization[name]
                getattr(q, name).zero_point = int(zp)
                getattr(q, name).scale = float(sc)
        return q


# ---- handles ---------------------------------------------------------------------------------
class Context:
    """WGPUContext analogue: one CUDA device."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        _check(lib().ws_context_create(int(device), C.byref(self._h)))
        self.device = int(device)

    @property
    def sm_count(self):
        return lib().ws_context_sm_count(self._h)

    def close(self):
        if getattr(self, "_h", None):
            lib().ws_context_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PointCloud:
    """pointcloud.rs:72-199."""

    def __init__(self):
        raise TypeError("use PointCloud.new(ctx, generic_pc)")

    @classmethod
    def new(cls, ctx, pc):
        self = object.__new__(cls)
        d = ws_pointcloud_desc()
        d.gaussians = pc.gaussians.ctypes.data
        d.num_points = pc.num_points
        d.sh_coefs = pc.sh_coefs.ctypes.data
        d.sh_bytes = pc.sh_coefs.nbytes
        q = pc.quantization_struct()
        if pc.compressed:
            d.covars = pc.covars.ctypes.data
            d.num_covars = pc.covars.nbytes // 12
            d.quantization = C.pointer(q)
        d.sh_deg, d.compressed = pc.sh_deg, int(pc.compressed)
        d.aabb = pc.aabb._c()
        d.center = _f3(pc.center)
        d.has_up = pc.up is not None
        if pc.up is not None:
            d.up = _f3(pc.up)
        d.has_mip_splatting = pc.mip_splatting is not None
        d.mip_splatting = bool(pc.mip_splatting)
        d.has_kernel_size = pc.kernel_size is not None
        d.kernel_size = float(pc.kernel_size or 0.0)
        d.has_background = pc.background_color is not None
        if pc.background_color is not None:
            d.background_color = _f3(pc.background_color)
        self._h = C.c_void_p()
        self._ctx = ctx
        _check(lib().ws_pointcloud_create(ctx._h, C.byref(d), C.byref(self._h)))
        return self

    @classmethod
    def from_ply(cls, ctx, file):
        """io/mod.rs:44-61 (`GenericGaussianPointCloud::load`) + PointCloud::new for a .ply: `file` is a
        path, a bytes-like object or a file object.  The vertex block is converted on the GPU."""
        if hasattr(file, "read"):
            data = file.read()
        elif isinstance(file, (bytes, bytearray, memoryview)):
            data = bytes(file)
        else:
            with open(file, "rb") as f:
                data = f.read()
        self = object.__new__(cls)
        self._h = C.c_void_p()
        self._ctx = ctx
        buf = np.frombuffer(data, dtype=np.uint8)
        _check(lib().ws_pointcloud_create_from_ply(ctx._h, buf.ctypes.data if len(buf) else None, len(buf), C.byref(self._h)))
        return self

    @classmethod
    def from_npz(cls, ctx, file):
        """io/mod.rs:53-58 + NpzReader (io/npz.rs:29-225) + PointCloud::new for a compressed .npz: `file` is a path,
        a file object, bytes, or a dict of the already-decoded members.  numpy decodes the zip/npy container;
        the arrays are assembled into the GPU layouts on the device."""
        if isinstance(file, dict):
            a = file
        else:
            if isinstance(file, (bytes, bytearray, memoryview)):
                import io
                file = io.BytesIO(bytes(file))
            with np.load(file) as z:
                a = {k: z[k] for k in z.files}
        keep = []

        def arr(name, dt, required=True):
            if a.get(name) is None:
                if required:
                    raise WsError(-1, "websplat_b200: invalid argument (status -1): array %r missing" % name)   # io/npz.rs:265-275
                return None
            v = np.ascontiguousarray(a[name], dtype=dt)
            keep.append(v)
            return v

        def scalar(name, default, cast):
            return cast(np.asarray(a[name]).reshape(-1)[0]) if a.get(name) is not None else default

        d = ws_c3dgs_arrays()
        xyz = arr("xyz", np.float16).reshape(-1, 3)
        opacity = arr("opacity", np.int8).reshape(-1)
        n = len(xyz)
        if len(opacity) != n:
            raise WsError(-1, "websplat_b200: invalid argument (status -1): opacity has %d entries for %d points" % (len(opacity), n))
        d.xyz, d.opacity, d.num_points = xyz.ctypes.data, opacity.ctypes.data, n
        has_sf = a.get("scaling_factor_scale") is not None                                      # io/npz.rs:88-96
        for name, dt in (("scaling_factor", np.int8), ("gaussian_indices", np.int32), ("feature_indices", np.int32)):
            v = arr(name, dt, required=(name == "scaling_factor" and has_sf))
            if name == "scaling_factor" and not has_sf:
                v = None
            if v is not None:
                if v.size != n:
                    raise WsError(-1, "websplat_b200: invalid argument (status -1): %s has %d entries for %d points" % (name, v.size, n))
                setattr(d, name, v.ctypes.data)
        scaling = arr("scaling", np.int8).reshape(-1, 3)
        rotation = arr("rotation", np.int8).reshape(-1, 4)
        if len(scaling) != len(rotation):
            raise WsError(-1, "websplat_b200: invalid argument (status -1): scaling / rotation lengths differ")
        d.scaling, d.rotation, d.num_covars = scaling.ctypes.data, rotation.ctypes.data, len(rotation)
        dc = arr("features_dc", np.int8).reshape(-1, 3)
        rest = arr("features_rest", np.int8)
        # sh degree from features_rest.shape[1] + 1 (io/npz.rs:33-37)
        ncoef = (rest.shape[1] + 1) if rest.ndim >= 2 else 1
        deg = int(round(ncoef ** 0.5)) - 1
        if (deg + 1) ** 2 != ncoef:
            raise WsError(-1, "websplat_b200: invalid argument (status -1): num sh coefs not valid")
        if rest.size != len(dc) * (ncoef - 1) * 3:
            raise WsError(-1, "websplat_b200: invalid argument (status -1): features_rest / features_dc lengths differ")
        d.features_dc, d.features_rest, d.num_features, d.sh_deg = dc.ctypes.data, rest.ctypes.data, len(dc), deg
        d.scaling_scale, d.scaling_zero_point = scalar("scaling_scale", 1.0, float), scalar("scaling_zero_point", 0, int)
        d.rotation_scale, d.rotation_zero_point = scalar("rotation_scale", 1.0, float), scalar("rotation_zero_point", 0, int)
        for field, key in (("color_dc", "features_dc"), ("color_rest", "features_rest"), ("opacity", "opacity"), ("scaling_factor", "scaling_factor")):
            qz = getattr(d.quantization, field)
            qz.zero_point = scalar(key + "_zero_point", 0, int) if (key != "scaling_factor" or has_sf) else 0
            qz.scale = scalar(key + "_scale", 1.0, float) if (key != "scaling_factor" or has_sf) else 1.0
        if a.get("mip_splatting") is not None:
            d.has_mip_splatting, d.mip_splatting = 1, int(bool(np.asarray(a["mip_splatting"]).reshape(-1)[0]))
        if a.get("kernel_size") is not None:
            d.has_kernel_size, d.kernel_size = 1, float(np.asarray(a["kernel_size"]).reshape(-1)[0])
        if a.get("background_color") is not None:
            d.has_background, d.background_color = 1, _f3(np.asarray(a["background_color"], np.float32).reshape(-1)[:3])
        self = object.__new__(cls)
        self._h = C.c_void_p()
        self._ctx = ctx
        _check(lib().ws_pointcloud_create_from_c3dgs(ctx._h, C.byref(d), C.byref(self._h)))
        return self

    def read(self, which):
        """Debug read-back of the resident layouts: 'gaussians' (n, 28|24) u8, 'sh_coefs' (n, 96) u8 (raw) or the flat
        i8 codebook (compressed), 'xyz' (n, 3) f32, 'covars' (K, 12) u8 (compressed)."""
        idx = {"gaussians": 0, "sh_coefs": 1, "xyz": 2, "covars": 3}[which]
        nbytes = lib().ws_pointcloud_buffer_bytes(self._h, idx)
        out = np.zeros(nbytes, np.uint8)
        _check(lib().ws_pointcloud_read(self._h, idx, out.ctypes.data, out.nbytes))
        if idx == 0:
            return out.reshape(-1, 24 if self.compressed() else 28)
        if idx == 1:
            return out.view(np.int8) if self.compressed() else out.reshape(-1, 96)
        if idx == 2:
            return out.view(np.float32).reshape(-1, 3)
        return out.reshape(-1, 12)

    def background_color(self):
        o = (C.c_float * 3)()
        return np.array(o[:], dtype=np.float32) if lib().ws_pointcloud_background_color(self._h, C.byref(o)) else None

    def num_points(self):
        return lib().ws_pointcloud_num_points(self._h)

    def sh_deg(self):
        return lib().ws_pointcloud_sh_deg(self._h)

    def compressed(self):
        return bool(lib().ws_pointcloud_compressed(self._h))

    def bbox(self):
        b = ws_aabb()
        _check(lib().ws_pointcloud_bbox(self._h, C.byref(b)))
        return Aabb(b.min[:], b.max[:])

    def center(self):
        o = (C.c_float * 3)()
        _check(lib().ws_pointcloud_center(self._h, C.byref(o)))
        return np.array(o[:], dtype=np.float32)

    def up(self):
        o = (C.c_float * 3)()
        return np.array(o[:], dtype=np.float32) if lib().ws_pointcloud_up(self._h, C.byref(o)) else None

    def mip_splatting(self):
        o = C.c_int32()
        return bool(o.value) if lib().ws_pointcloud_mip_splatting(self._h, C.byref(o)) else None

    def dilation_kernel_size(self):
        o = C.c_float()
        return o.value if lib().ws_pointcloud_dilation_kernel_size(self._h, C.byref(o)) else None

    def close(self):
        if getattr(self, "_h", None):
            lib().ws_pointcloud_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _stream_handle(stream):
    if stream is None:
        return None
    if isinstance(stream, int):
        return C.c_void_p(stream)
    return C.c_void_p(int(stream.cuda_stream))     # torch.cuda.Stream


class GaussianRenderer:
    """renderer.rs:17-288."""

    def __init__(self):
        raise TypeError("use GaussianRenderer.new(ctx, color_format, sh_deg, compressed)")

    @classmethod
    def new(cls, ctx, color_format, sh_deg, compressed):
        self = object.__new__(cls)
        self._h = C.c_void_p()
        self._ctx = ctx
        self._format = int(color_format)
        self._viewport = None
        _check(lib().ws_renderer_create(ctx._h, int(color_format), int(sh_deg), int(bool(compressed)), C.byref(self._h)))
        return self

    def color_format(self):
        return lib().ws_renderer_color_format(self._h)

    def set_pair_capacity(self, max_pairs):
        _check(lib().ws_renderer_set_pair_capacity(self._h, int(max_pairs)))

    def set_timing(self, enabled):
        _check(lib().ws_renderer_set_timing(self._h, int(bool(enabled))))

    def set_occlusion_split(self, enabled):
        """Two depth slabs with saturated-tile culling of the far one (bit-identical image, fewer pairs).
        True / False, or None for the default: automatic (on from 2 M points)."""
        _check(lib().ws_renderer_set_occlusion_split(self._h, -1 if enabled is None else int(bool(enabled))))

    def set_cuda_graphs(self, enabled):
        _check(lib().ws_renderer_set_cuda_graphs(self._h, int(bool(enabled))))

    def prepare(self, stream, pc, render_settings):
        """Enqueue stage 1 + 2 on `stream` (torch.cuda.Stream, raw cudaStream_t int, or None)."""
        a = render_settings._c()
        self._viewport = render_settings.viewport
        _check(lib().ws_renderer_prepare(self._h, pc._h, C.byref(a), _stream_handle(stream)))

    def render(self, target, pc, clear=(0.0, 0.0, 0.0, 0.0), stream=None, row_pitch=None):
        """Enqueue stage 3 into `target`: a device pointer (int) or an object with .data_ptr()
        (a CUDA torch tensor of H x W x 4 in the renderer's format)."""
        ptr = target if isinstance(target, int) else target.data_ptr()
        if row_pitch is None:
            row_pitch = self._viewport[0] * _BPP[self._format]
        clr = (C.c_double * 4)(*[float(c) for c in clear])
        _check(lib().ws_renderer_render(self._h, pc._h, C.c_void_p(ptr), row_pitch, C.byref(clr), _stream_handle(stream)))

    def render_to_host(self, host_target, pc, clear=(0.0, 0.0, 0.0, 0.0), stream=None):
        """render + download_texture (bin/render.rs:187-246) into host memory: a numpy array or a
        (pinned) CPU torch tensor of H x W x 4.  Asynchronous on `stream`; synchronise before reading."""
        ptr = host_target.ctypes.data if isinstance(host_target, np.ndarray) else host_target.data_ptr()
        row_pitch = self._viewport[0] * _BPP[self._format]
        clr = (C.c_double * 4)(*[float(c) for c in clear])
        _check(lib().ws_renderer_render_to_host(self._h, pc._h, C.c_void_p(ptr), row_pitch, C.byref(clr), _stream_handle(stream)))

    def prepare_views(self, stream, pc, render_settings):
        """Enqueue stage 1 + 2 for a batch of up to MAX_VIEWS views of `pc` (a list of SplattingArgs with one viewport).
        Every view renders bit-identical to the same view through prepare + render."""
        args = list(render_settings)
        arr = (ws_splatting_args * max(len(args), 1))(*[a._c() for a in args])
        self._viewport = args[0].viewport if args else self._viewport
        self._views = len(args)
        _check(lib().ws_renderer_prepare_views(self._h, pc._h, arr, len(args), _stream_handle(stream)))

    def render_views(self, target, pc, clear=(0.0, 0.0, 0.0, 0.0), stream=None, row_pitch=None, view_stride=None):
        """Enqueue stage 3 of the batch into `target`: a device pointer (int) or a CUDA torch tensor of K x H x W x 4
        in the renderer's format; view v starts `view_stride` bytes after view v - 1 (default: H * row_pitch)."""
        ptr = target if isinstance(target, int) else target.data_ptr()
        if row_pitch is None:
            row_pitch = self._viewport[0] * _BPP[self._format]
        if view_stride is None:
            view_stride = self._viewport[1] * row_pitch
        clr = (C.c_double * 4)(*[float(c) for c in clear])
        _check(lib().ws_renderer_render_views(self._h, pc._h, C.c_void_p(ptr), row_pitch, view_stride, C.byref(clr), _stream_handle(stream)))

    def render_views_to_host(self, host_target, pc, clear=(0.0, 0.0, 0.0, 0.0), stream=None):
        """render_views into host memory: a numpy array or a (pinned) CPU torch tensor of K x H x W x 4.  Asynchronous
        on `stream`; synchronise before reading."""
        ptr = host_target.ctypes.data if isinstance(host_target, np.ndarray) else host_target.data_ptr()
        row_pitch = self._viewport[0] * _BPP[self._format]
        clr = (C.c_double * 4)(*[float(c) for c in clear])
        _check(lib().ws_renderer_render_views_to_host(self._h, pc._h, C.c_void_p(ptr), row_pitch, self._viewport[1] * row_pitch,
                                                      C.byref(clr), _stream_handle(stream)))

    def views_num_visible_points(self):
        """Per-view visible point counts of the last batch (synchronises)."""
        k = getattr(self, "_views", 0)
        o = (C.c_uint32 * max(k, 1))()
        _check(lib().ws_renderer_views_num_visible_points(self._h, o, k))
        return [int(x) for x in o[:k]]

    def empty_host_frame(self):
        dt, ch = _NP_PIXEL[self._format]
        return np.empty((self._viewport[1], self._viewport[0], ch), dtype=dt)

    def num_visible_points(self):
        o = C.c_uint32()
        _check(lib().ws_renderer_num_visible_points(self._h, C.byref(o)))
        return o.value

    def stats(self, allow_overflow=False):
        s = ws_frame_stats()
        st = lib().ws_renderer_stats(self._h, C.byref(s))
        if st != WS_OK and not (allow_overflow and st == WS_ERR_PAIR_OVERFLOW):
            _check(st)
        out = {name: getattr(s, name) for name, _ in ws_frame_stats._fields_}
        out["pair_overflow"] = (st == WS_ERR_PAIR_OVERFLOW)
        return out

    def read_buffer(self, which):
        """Intermediate buffers of the last prepared frame (parity tests)."""
        need = C.c_size_t()
        dummy = (C.c_uint8 * 8)()
        st = lib().ws_renderer_read_buffer(self._h, which, C.cast(dummy, C.c_void_p), 0, C.byref(need))
        if st != WS_OK and need.value == 0:
            _check(st)
        buf = np.empty(max(need.value, 1), dtype=np.uint8)
        if need.value:
            _check(lib().ws_renderer_read_buffer(self._h, which, C.c_void_p(buf.ctypes.data), need.value, C.byref(need)))
        buf = buf[:need.value]
        if which == BUF_SPLATS_2D:
            return buf.view(np.uint16).reshape(-1, 10)
        if which == BUF_TILE_RECTS:
            return buf.view(np.uint16).reshape(-1, 4)       # x0, y0, w, h
        if which == BUF_TILE_RANGES:
            return buf.view(np.uint32).reshape(-1, 2)
        return buf.view(np.uint32)

    def camera_uniform(self):
        o = (C.c_float * 68)()
        _check(lib().ws_renderer_camera_uniform(self._h, C.byref(o)))
        return np.array(o[:], dtype=np.float32)

    def settings_uniform(self):
        buf = np.zeros(80, dtype=np.uint8)
        _check(lib().ws_renderer_settings_uniform(self._h, C.c_void_p(buf.ctypes.data)))
        return buf

    def close(self):
        if getattr(self, "_h", None):
            lib().ws_renderer_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def ply_probe(data):
    """Header-only parse of a .ply image (io/ply.rs:28-48); host code, no GPU needed."""
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    info = ws_ply_info()
    _check(lib().ws_ply_probe(buf.ctypes.data if len(buf) else None, len(buf), C.byref(info)))
    return dict(num_points=info.num_points, data_offset=info.data_offset, sh_deg=info.sh_deg, stride_bytes=info.stride_bytes,
                big_endian=bool(info.big_endian),
                mip_splatting=bool(info.mip_splatting) if info.has_mip_splatting else None,
                kernel_size=info.kernel_size if info.has_kernel_size else None,
                background_color=list(info.background_color) if info.has_background else None)


def sort_pairs_host(ctx, keys, payload, key_bits=32):
    """GPURSSorter::record_sort on host arrays (gpu_rs.rs:865-873): stable ascending, in place."""
    keys = np.ascontiguousarray(keys, dtype=np.uint32)
    payload = np.ascontiguousarray(payload, dtype=np.uint32)
    assert keys.shape == payload.shape and keys.ndim == 1
    _check(lib().ws_sort_pairs_u32_host(ctx._h, C.c_void_p(keys.ctypes.data), C.c_void_p(payload.ctypes.data),
                                        keys.size, int(key_bits)))
    return keys, payload


from . import scene, synth  # noqa: E402,F401
from .scene import Scene, SceneCamera  # noqa: E402,F401
from .distributed import ShardedPipeline, ShardedRenderer, balanced_bands, shard_cloud, tile_row_bands  # noqa: E402,F401
