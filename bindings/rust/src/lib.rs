//! Drop-in for web-splat's render path on a B200: the reference's `PointCloud`, `SplattingArgs` and
//! `GaussianRenderer::{new, prepare, render, num_visible_points, color_format}` (src/pointcloud.rs:72-349,
//! src/renderer.rs:33-260,587-599) on top of libwebsplat_b200.so.  SOURCE ONLY -- see Cargo.toml.
//!
//! Differences a caller sees (INTEGRATION.md section 3): `wgpu::Device/Queue` -> `&Context`; the command encoder ->
//! a CUDA stream handle; the render pass' colour attachment -> a device (or host) pixel buffer + the clear colour.
pub mod ffi;

use anyhow::{anyhow, Result};
use cgmath::{Point3, Quaternion, Vector2, Vector3};
use std::ffi::CStr;
use std::os::raw::c_void;
use std::time::Duration;

fn check(status: i32) -> Result<()> {
    if status == ffi::WS_OK {
        return Ok(());
    }
    let (what, detail) = unsafe {
        (CStr::from_ptr(ffi::ws_status_string(status)).to_string_lossy().into_owned(),
         CStr::from_ptr(ffi::ws_last_error()).to_string_lossy().into_owned())
    };
    Err(anyhow!("websplat_b200: {what} (status {status}): {detail}"))
}

/// `WGPUContext::new_instance()` (src/lib.rs:69): one CUDA device.
pub struct Context { h: *mut ffi::ws_context }
impl Context {
    pub fn new(cuda_device: i32) -> Result<Self> {
        let mut h = std::ptr::null_mut();
        check(unsafe { ffi::ws_context_create(cuda_device, &mut h) })?;
        Ok(Self { h })
    }
}
impl Drop for Context { fn drop(&mut self) { unsafe { ffi::ws_context_destroy(self.h) } } }

/// A CUDA stream owned by the caller (`cudaStream_t`), the analogue of the caller's command encoder.
#[derive(Copy, Clone)]
pub struct Stream(pub *mut c_void);
impl Stream { pub fn default_stream() -> Self { Stream(std::ptr::null_mut()) } }

#[derive(Copy, Clone, Debug)]
pub struct Aabb { pub min: Point3<f32>, pub max: Point3<f32> }
impl From<Aabb> for ffi::ws_aabb { fn from(b: Aabb) -> Self { ffi::ws_aabb { min: b.min.into(), max: b.max.into() } } }

/// `PerspectiveProjection` (src/camera.rs:86-94) and `PerspectiveCamera` (src/camera.rs:7-11), field for field.
#[derive(Copy, Clone, Debug)]
pub struct PerspectiveProjection { pub fovx: f32, pub fovy: f32, pub znear: f32, pub zfar: f32, pub fov2view_ratio: f32 }
#[derive(Copy, Clone, Debug)]
pub struct PerspectiveCamera { pub position: Point3<f32>, pub rotation: Quaternion<f32>, pub projection: PerspectiveProjection }
impl PerspectiveCamera {
    /// `fit_near_far` (src/camera.rs:26-35).
    pub fn fit_near_far(&mut self, aabb: &Aabb) {
        let pos: [f32; 3] = self.position.into();
        let b: ffi::ws_aabb = (*aabb).into();
        unsafe { ffi::ws_camera_fit_near_far(pos.as_ptr(), &b, &mut self.projection.znear, &mut self.projection.zfar) }
    }
}

/// `SplattingArgs` (src/renderer.rs:587-599), same fields, same `Option`s.
#[derive(Clone, Debug)]
pub struct SplattingArgs {
    pub camera: PerspectiveCamera,
    pub viewport: Vector2<u32>,
    pub gaussian_scaling: f32,
    pub max_sh_deg: u32,
    pub mip_splatting: Option<bool>,
    pub kernel_size: Option<f32>,
    pub clipping_box: Option<Aabb>,
    pub walltime: Duration,
    pub scene_center: Option<Point3<f32>>,
    pub scene_extend: Option<f32>,
    pub background_color: [f64; 4],
}
impl From<&SplattingArgs> for ffi::ws_splatting_args {
    fn from(a: &SplattingArgs) -> Self {
        let q = a.camera.rotation;
        let p = a.camera.projection;
        let mut o = ffi::ws_splatting_args::default();
        o.cam_position = a.camera.position.into();
        o.cam_rotation_wxyz = [q.s, q.v.x, q.v.y, q.v.z];
        o.fovx = p.fovx; o.fovy = p.fovy; o.znear = p.znear; o.zfar = p.zfar; o.fov2view_ratio = p.fov2view_ratio;
        o.viewport = [a.viewport.x, a.viewport.y];
        o.gaussian_scaling = a.gaussian_scaling;
        o.max_sh_deg = a.max_sh_deg;
        if let Some(m) = a.mip_splatting { o.has_mip_splatting = 1; o.mip_splatting = m as i32; }
        if let Some(k) = a.kernel_size { o.has_kernel_size = 1; o.kernel_size = k; }
        if let Some(b) = a.clipping_box { o.has_clipping_box = 1; o.clipping_box = b.into(); }
        o.walltime_secs = a.walltime.as_secs_f32();                    // src/renderer.rs:643
        if let Some(c) = a.scene_center { o.has_scene_center = 1; o.scene_center = c.into(); }
        if let Some(e) = a.scene_extend { o.has_scene_extend = 1; o.scene_extend = e; }
        o.background_color = a.background_color;
        o
    }
}

/// `PointCloud` (src/pointcloud.rs:72-349).  `new` takes the CPU byte buffers of a `GenericGaussianPointCloud`
/// (src/io/mod.rs:27-42) through `ws_pointcloud_desc`; `from_ply` converts the file on the GPU instead.
pub struct PointCloud { h: *mut ffi::ws_pointcloud }
impl PointCloud {
    /// # Safety
    /// the pointers in `desc` must be valid for the sizes it states for the duration of the call.
    pub unsafe fn new(ctx: &Context, desc: &ffi::ws_pointcloud_desc) -> Result<Self> {
        let mut h = std::ptr::null_mut();
        check(ffi::ws_pointcloud_create(ctx.h, desc, &mut h))?;
        Ok(Self { h })
    }
    pub fn from_ply(ctx: &Context, file: &[u8]) -> Result<Self> {
        let mut h = std::ptr::null_mut();
        check(unsafe { ffi::ws_pointcloud_create_from_ply(ctx.h, file.as_ptr() as *const c_void, file.len() as u64, &mut h) })?;
        Ok(Self { h })
    }
    pub fn num_points(&self) -> u32 { unsafe { ffi::ws_pointcloud_num_points(self.h) } }
    pub fn sh_deg(&self) -> u32 { unsafe { ffi::ws_pointcloud_sh_deg(self.h) } }
    pub fn compressed(&self) -> bool { unsafe { ffi::ws_pointcloud_compressed(self.h) != 0 } }
    pub fn bbox(&self) -> Aabb {
        let mut b = ffi::ws_aabb::default();
        unsafe { ffi::ws_pointcloud_bbox(self.h, &mut b) };
        Aabb { min: b.min.into(), max: b.max.into() }
    }
    pub fn center(&self) -> Point3<f32> {
        let mut c = [0f32; 3];
        unsafe { ffi::ws_pointcloud_center(self.h, c.as_mut_ptr()) };
        c.into()
    }
    pub fn up(&self) -> Option<Vector3<f32>> {
        let mut u = [0f32; 3];
        (unsafe { ffi::ws_pointcloud_up(self.h, u.as_mut_ptr()) } != 0).then(|| u.into())
    }
    pub fn mip_splatting(&self) -> Option<bool> {
        let mut v = 0i32;
        (unsafe { ffi::ws_pointcloud_mip_splatting(self.h, &mut v) } != 0).then_some(v != 0)
    }
    pub fn dilation_kernel_size(&self) -> Option<f32> {
        let mut v = 0f32;
        (unsafe { ffi::ws_pointcloud_dilation_kernel_size(self.h, &mut v) } != 0).then_some(v)
    }
}
impl Drop for PointCloud { fn drop(&mut self) { unsafe { ffi::ws_pointcloud_destroy(self.h) } } }

/// The three `wgpu::TextureFormat`s the reference's callers use (src/lib.rs:192-196, bin/render.rs:154, bin/video.rs:186).
#[derive(Copy, Clone, Debug, PartialEq, Eq)]
pub enum ColorFormat { Rgba8Unorm = 0, Rgba16Float = 1, Rgba32Float = 2 }
impl ColorFormat { pub fn bytes_per_pixel(self) -> usize { match self { Self::Rgba8Unorm => 4, Self::Rgba16Float => 8, Self::Rgba32Float => 16 } } }

/// `GaussianRenderer` (src/renderer.rs:20-31).  Not re-entrant, like `&mut self` upstream.
pub struct GaussianRenderer { h: *mut ffi::ws_renderer, format: ColorFormat, views: u32 }
impl GaussianRenderer {
    /// `GaussianRenderer::new` (src/renderer.rs:33).
    pub fn new(ctx: &Context, color_format: ColorFormat, sh_deg: u32, compressed: bool) -> Result<Self> {
        let mut h = std::ptr::null_mut();
        check(unsafe { ffi::ws_renderer_create(ctx.h, color_format as i32, sh_deg, compressed as i32, &mut h) })?;
        Ok(Self { h, format: color_format, views: 0 })
    }
    /// `prepare` (src/renderer.rs:191): enqueues stage 1 + 2 on `stream`.
    ///
    /// Everything is asynchronous, so a frame that turns out incomplete on the device (pair capacity exceeded, internal
    /// error flag) cannot fail the call that enqueued it: the NEXT `prepare` that finds the earlier frame's status copy
    /// completed returns that frame's error once (`PairOverflow` / `Cuda`) and enqueues nothing; calling it again proceeds.
    /// `stats()` reports (and consumes) the status of the frame it synchronises.
    pub fn prepare(&mut self, stream: Stream, pc: &PointCloud, render_settings: &SplattingArgs) -> Result<()> {
        let a = ffi::ws_splatting_args::from(render_settings);
        check(unsafe { ffi::ws_renderer_prepare(self.h, pc.h, &a, stream.0) })
    }
    /// `render` (src/renderer.rs:250) + the caller's `LoadOp::Clear(clear)`: stage 3 into device memory.
    ///
    /// # Safety
    /// `target_device` must point at `height * row_pitch` bytes of device memory of the renderer's colour format.
    pub unsafe fn render(&self, stream: Stream, pc: &PointCloud, target_device: *mut c_void, row_pitch: usize, clear: [f64; 4]) -> Result<()> {
        check(ffi::ws_renderer_render(self.h, pc.h, target_device, row_pitch, clear.as_ptr(), stream.0))
    }
    /// render + `download_texture` (bin/render.rs:187-246): the frame lands in `target_host` (asynchronously on `stream`).
    pub fn render_to_host(&self, stream: Stream, pc: &PointCloud, target_host: &mut [u8], width: u32, clear: [f64; 4]) -> Result<()> {
        let pitch = width as usize * self.format.bytes_per_pixel();
        check(unsafe { ffi::ws_renderer_render_to_host(self.h, pc.h, target_host.as_mut_ptr() as *mut c_void, pitch, clear.as_ptr(), stream.0) })
    }
    /// `num_visible_points` (src/renderer.rs:170): blocking read-back of V.
    pub fn num_visible_points(&self) -> Result<u32> {
        let mut v = 0u32;
        check(unsafe { ffi::ws_renderer_num_visible_points(self.h, &mut v) })?;
        Ok(v)
    }
    /// A batch of up to `ffi::WS_MAX_VIEWS` views of one cloud (one viewport): stage 1 + 2 for all of them. Every view
    /// renders bit-identical to the same view through `prepare` + `render`.
    pub fn prepare_views(&mut self, stream: Stream, pc: &PointCloud, render_settings: &[SplattingArgs]) -> Result<()> {
        let a: Vec<ffi::ws_splatting_args> = render_settings.iter().map(ffi::ws_splatting_args::from).collect();
        check(unsafe { ffi::ws_renderer_prepare_views(self.h, pc.h, a.as_ptr(), a.len() as u32, stream.0) })?;
        self.views = a.len() as u32;
        Ok(())
    }
    /// Stage 3 of the batch into device memory: view v starts at `target_device + v * view_stride`.
    ///
    /// # Safety
    /// `target_device` must point at `views * view_stride` bytes of device memory of the renderer's colour format.
    pub unsafe fn render_views(&self, stream: Stream, pc: &PointCloud, target_device: *mut c_void, row_pitch: usize, view_stride: usize,
                               clear: [f64; 4]) -> Result<()> {
        check(ffi::ws_renderer_render_views(self.h, pc.h, target_device, row_pitch, view_stride, clear.as_ptr(), stream.0))
    }
    /// The batch into `target_host`, tightly packed: view v at byte `v * width * height * bytes_per_pixel`
    /// (asynchronously on `stream`).
    pub fn render_views_to_host(&self, stream: Stream, pc: &PointCloud, target_host: &mut [u8], width: u32, height: u32, clear: [f64; 4]) -> Result<()> {
        let pitch = width as usize * self.format.bytes_per_pixel();
        let stride = pitch * height as usize;
        if target_host.len() < stride * self.views as usize {
            return Err(anyhow!("websplat_b200: host buffer smaller than the batch"));
        }
        check(unsafe { ffi::ws_renderer_render_views_to_host(self.h, pc.h, target_host.as_mut_ptr() as *mut c_void, pitch, stride, clear.as_ptr(), stream.0) })
    }
    /// Per-view visible point counts of the last batch (blocking).
    pub fn views_num_visible_points(&self) -> Result<Vec<u32>> {
        let mut v = vec![0u32; self.views as usize];
        check(unsafe { ffi::ws_renderer_views_num_visible_points(self.h, v.as_mut_ptr(), self.views) })?;
        Ok(v)
    }
    /// The `GPUStopwatch` replacement: "preprocess" / "sorting" / "rasterization" (src/renderer.rs:220-239) as ms.
    pub fn stats(&self) -> Result<ffi::ws_frame_stats> {
        let mut s = ffi::ws_frame_stats::default();
        check(unsafe { ffi::ws_renderer_stats(self.h, &mut s) })?;
        Ok(s)
    }
    pub fn color_format(&self) -> ColorFormat { self.format }
}
impl Drop for GaussianRenderer { fn drop(&mut self) { unsafe { ffi::ws_renderer_destroy(self.h) } } }
