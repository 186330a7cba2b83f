//! Raw bindings to include/rtrace.h (the subset the host needs).
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct RtScene {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtCamera {
    pub eye: [f32; 3],
    pub right: [f32; 3],
    pub up: [f32; 3],
    pub forward: [f32; 3],
}

#[repr(C)]
#[derive(Default, Clone, Copy)]
pub struct RtStats {
    pub primary_rays: u64,
    pub shadow_rays: u64,
    pub kernel_ms: f64,
    pub total_ms: f64,
    pub kernel_launches: u32,
    pub gpus: u32,
    pub variant_used: u32,
    pub reserved: u32,
}

pub type RtFrameCallback = extern "C" fn(user: *mut c_void, frame: u32, rgba: *const u8, len: usize);
/// Fills `camera_out` (or sets `*use_camera = 0` for the reference camera) and returns the frame id, or -1.
pub type RtNextFrameCallback = extern "C" fn(user: *mut c_void, camera_out: *mut RtCamera, use_camera: *mut c_int) -> c_int;

extern "C" {
    pub fn rt_last_error() -> *const c_char;
    pub fn rt_set_device(device: c_int) -> c_int;
    pub fn rt_scene_create(level: u32, origin: *const f32, radius: f32, light: *const f32, eye: *const f32,
                           out: *mut *mut RtScene) -> c_int;
    pub fn rt_scene_destroy(s: *mut RtScene);
    pub fn rt_scene_counts(s: *const RtScene, groups: *mut u64, items: *mut u64) -> c_int;
    pub fn rt_render_region(s: *const RtScene, width: u16, height: u16, spp: u16, l: u16, b: u16, r: u16, t: u16,
                            rgba_out: *mut u8, rgba_len: usize) -> c_int;
    pub fn rt_render_preview(s: *const RtScene, camera: *const RtCamera, width: u32, height: u32, step: u32,
                             rgba_out: *mut u8, rgba_len: usize, stream: *mut c_void) -> c_int;
    pub fn rt_render_frame_multi(scenes: *const *mut RtScene, ngpu: c_int, camera: *const RtCamera, width: u32,
                                 height: u32, spp: u32, rgba_out: *mut u8, rgba_len: usize, stats: *mut RtStats) -> c_int;
    // the frame before quantisation: {r, g, b, alpha} as f32, 16 bytes per pixel (include/rtrace.h "float output")
    pub fn rt_render_frame_multi_f32(scenes: *const *mut RtScene, ngpu: c_int, camera: *const RtCamera, width: u32,
                                     height: u32, spp: u32, rgba_out: *mut f32, rgba_bytes: usize,
                                     stats: *mut RtStats) -> c_int;
    pub fn rt_render_sweep(s: *const RtScene, cameras: *const RtCamera, n_frames: u32, width: u32, height: u32,
                           spp: u32, cb: RtFrameCallback, user: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_sweep_rgb(s: *const RtScene, cameras: *const RtCamera, n_frames: u32, width: u32, height: u32,
                               spp: u32, cb: RtFrameCallback, user: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_sweep_pull(s: *const RtScene, next: RtNextFrameCallback, next_user: *mut c_void, width: u32,
                                height: u32, spp: u32, rgb: c_int, cb: RtFrameCallback, user: *mut c_void,
                                stats: *mut RtStats) -> c_int;
    pub fn rt_render_sweep_multi(scenes: *const *mut RtScene, ngpu: c_int, cameras: *const RtCamera, n_frames: u32,
                                 width: u32, height: u32, spp: u32, rgb: c_int, cb: RtFrameCallback,
                                 user: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_rows(s: *const RtScene, camera: *const RtCamera, width: u32, height: u32, spp: u32,
                          row_start: u32, row_stride: u32, row_count: u32, rgba_out: *mut u8, pitch_bytes: usize,
                          kinds_out: *mut u8, stream: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_rows_f32(s: *const RtScene, camera: *const RtCamera, width: u32, height: u32, spp: u32,
                              row_start: u32, row_stride: u32, row_count: u32, rgba_out: *mut f32, pitch_bytes: usize,
                              stream: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_row_blocks(s: *const RtScene, camera: *const RtCamera, width: u32, height: u32, spp: u32,
                                row_start: u32, row_stride: u32, row_block: u32, row_count: u32, rgba_out: *mut u8,
                                pitch_bytes: usize, absolute_rows: c_int, stream: *mut c_void,
                                stats: *mut RtStats) -> c_int;
    pub fn rt_host_alloc(bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn rt_host_free(p: *mut c_void);
    pub fn rt_png_bound(width: u32, height: u32, bytes: *mut usize) -> c_int;
    pub fn rt_encode_png(rgba: *const u8, width: u32, height: u32, pitch_bytes: usize, png_out: *mut u8, cap: usize,
                         len_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn rt_render_sweep_png(scenes: *const *mut RtScene, ngpu: c_int, cameras: *const RtCamera, n_frames: u32,
                               width: u32, height: u32, spp: u32, cb: RtFrameCallback, user: *mut c_void,
                               stats: *mut RtStats) -> c_int;
    pub fn rt_apng_bound(width: u32, height: u32, n_frames: u32, frame_bytes: *mut usize) -> c_int;
    pub fn rt_encode_apng_frame(rgba: *const u8, width: u32, height: u32, pitch_bytes: usize, frame: u32,
                                n_frames: u32, delay_num: u16, delay_den: u16, out: *mut u8, cap: usize,
                                len_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn rt_render_sweep_apng(scenes: *const *mut RtScene, ngpu: c_int, cameras: *const RtCamera, n_frames: u32,
                                width: u32, height: u32, spp: u32, delay_num: u16, delay_den: u16,
                                cb: RtFrameCallback, user: *mut c_void, stats: *mut RtStats) -> c_int;
}

pub fn last_error() -> String {
    unsafe { std::ffi::CStr::from_ptr(rt_last_error()) }.to_string_lossy().into_owned()
}
