//! Raw declarations, one to one with include/websplat_b200.h (same field order, same widths).
#![allow(non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_int, c_void};

pub const WS_OK: i32 = 0;
pub const WS_ERR_PAIR_OVERFLOW: i32 = -4;
pub const WS_MAX_VIEWS: usize = 8;

#[repr(C)] #[derive(Copy, Clone, Default, Debug)] pub struct ws_aabb { pub min: [f32; 3], pub max: [f32; 3] }
#[repr(C)] #[derive(Copy, Clone, Default)] pub struct ws_quantization { pub zero_point: i32, pub scale: f32, pub _pad: [u32; 2] }
#[repr(C)] #[derive(Copy, Clone, Default)]
pub struct ws_quantization4 { pub color_dc: ws_quantization, pub color_rest: ws_quantization, pub opacity: ws_quantization, pub scaling_factor: ws_quantization }

#[repr(C)]
pub struct ws_pointcloud_desc {
    pub gaussians: *const c_void, pub num_points: u64,
    pub sh_coefs: *const c_void, pub sh_bytes: u64,
    pub covars: *const c_void, pub num_covars: u64,
    pub quantization: *const ws_quantization4,
    pub sh_deg: u32, pub compressed: u32,
    pub aabb: ws_aabb, pub center: [f32; 3],
    pub has_up: i32, pub up: [f32; 3],
    pub has_mip_splatting: i32, pub mip_splatting: i32,
    pub has_kernel_size: i32, pub kernel_size: f32,
    pub has_background: i32, pub background_color: [f32; 3],
}

#[repr(C)] #[derive(Copy, Clone, Default)]
pub struct ws_splatting_args {
    pub cam_position: [f32; 3], pub cam_rotation_wxyz: [f32; 4],
    pub fovx: f32, pub fovy: f32, pub znear: f32, pub zfar: f32, pub fov2view_ratio: f32,
    pub viewport: [u32; 2], pub gaussian_scaling: f32, pub max_sh_deg: u32,
    pub has_mip_splatting: i32, pub mip_splatting: i32,
    pub has_kernel_size: i32, pub kernel_size: f32,
    pub has_clipping_box: i32, pub clipping_box: ws_aabb,
    pub walltime_secs: f32,
    pub has_scene_center: i32, pub scene_center: [f32; 3],
    pub has_scene_extend: i32, pub scene_extend: f32,
    pub background_color: [f64; 4],
}

#[repr(C)] #[derive(Copy, Clone, Default, Debug)]
pub struct ws_frame_stats {
    pub num_points: u32, pub num_visible: u32, pub num_pairs: u64, pub pair_capacity: u64,
    pub num_tiles: u32, pub width: u32, pub height: u32,
    pub ms_preprocess: f32, pub ms_sort: f32, pub ms_blend: f32,
    pub ms_depth_sort: f32, pub ms_binning: f32, pub ms_tile_sort: f32, pub ms_ranges: f32,
    pub bytes_preprocess: u64, pub bytes_sort: u64, pub bytes_blend: u64,
}

pub enum ws_context {}
pub enum ws_pointcloud {}
pub enum ws_renderer {}

extern "C" {
    pub fn ws_status_string(s: i32) -> *const c_char;
    pub fn ws_last_error() -> *const c_char;
    pub fn ws_context_create(cuda_device: c_int, out: *mut *mut ws_context) -> i32;
    pub fn ws_context_destroy(ctx: *mut ws_context);
    pub fn ws_pointcloud_create(ctx: *mut ws_context, desc: *const ws_pointcloud_desc, out: *mut *mut ws_pointcloud) -> i32;
    pub fn ws_pointcloud_create_from_ply(ctx: *mut ws_context, file_bytes: *const c_void, file_len: u64, out: *mut *mut ws_pointcloud) -> i32;
    pub fn ws_pointcloud_destroy(pc: *mut ws_pointcloud);
    pub fn ws_pointcloud_num_points(pc: *const ws_pointcloud) -> u32;
    pub fn ws_pointcloud_sh_deg(pc: *const ws_pointcloud) -> u32;
    pub fn ws_pointcloud_compressed(pc: *const ws_pointcloud) -> i32;
    pub fn ws_pointcloud_bbox(pc: *const ws_pointcloud, out: *mut ws_aabb) -> i32;
    pub fn ws_pointcloud_center(pc: *const ws_pointcloud, out: *mut f32) -> i32;
    pub fn ws_pointcloud_up(pc: *const ws_pointcloud, out: *mut f32) -> i32;
    pub fn ws_pointcloud_mip_splatting(pc: *const ws_pointcloud, out: *mut i32) -> i32;
    pub fn ws_pointcloud_dilation_kernel_size(pc: *const ws_pointcloud, out: *mut f32) -> i32;
    pub fn ws_camera_fit_near_far(position: *const f32, aabb: *const ws_aabb, znear: *mut f32, zfar: *mut f32);
    pub fn ws_renderer_create(ctx: *mut ws_context, format: c_int, sh_deg: u32, compressed: i32, out: *mut *mut ws_renderer) -> i32;
    pub fn ws_renderer_destroy(r: *mut ws_renderer);
    pub fn ws_renderer_prepare(r: *mut ws_renderer, pc: *mut ws_pointcloud, args: *const ws_splatting_args, stream: *mut c_void) -> i32;
    pub fn ws_renderer_render(r: *mut ws_renderer, pc: *mut ws_pointcloud, dst_device: *mut c_void, row_pitch: usize, clear: *const f64, stream: *mut c_void) -> i32;
    pub fn ws_renderer_render_to_host(r: *mut ws_renderer, pc: *mut ws_pointcloud, dst_host: *mut c_void, row_pitch: usize, clear: *const f64, stream: *mut c_void) -> i32;
    pub fn ws_renderer_num_visible_points(r: *mut ws_renderer, out: *mut u32) -> i32;
    pub fn ws_renderer_prepare_views(r: *mut ws_renderer, pc: *mut ws_pointcloud, args: *const ws_splatting_args, num_views: u32, stream: *mut c_void) -> i32;
    pub fn ws_renderer_render_views(r: *mut ws_renderer, pc: *mut ws_pointcloud, dst_device: *mut c_void, row_pitch: usize, view_stride: usize, clear: *const f64, stream: *mut c_void) -> i32;
    pub fn ws_renderer_render_views_to_host(r: *mut ws_renderer, pc: *mut ws_pointcloud, dst_host: *mut c_void, row_pitch: usize, view_stride: usize, clear: *const f64, stream: *mut c_void) -> i32;
    pub fn ws_renderer_views_num_visible_points(r: *mut ws_renderer, out: *mut u32, count: u32) -> i32;
    pub fn ws_renderer_stats(r: *mut ws_renderer, out: *mut ws_frame_stats) -> i32;
    pub fn ws_renderer_set_pair_capacity(r: *mut ws_renderer, max_pairs: u64) -> i32;
}
