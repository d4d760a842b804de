//! Raw bindings to `include/raingun_b200.h` (ABI version 1).  Field order and types mirror the C
//! structs exactly; see the header for the meaning of every field and the reference lines each
//! entry point replaces.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const RG_ABI_VERSION: u32 = 2;
pub const RG_MAX_DEPTH: u32 = 64;
pub const RG_MAX_LIGHTS: u32 = 32; // obsolete: any light count is accepted (the size of one light chunk)
pub const RG_IPC_HANDLE_BYTES: usize = 64;

pub const RG_OK: c_int = 0;
pub const RG_E_INVALID: c_int = -1;
pub const RG_E_PORTRAIT: c_int = -2; // assert!(width >= height), ray.rs:42
pub const RG_E_TOO_LARGE: c_int = -3; // u32 width * height, rendering.rs:27
pub const RG_E_DEPTH: c_int = -4;
pub const RG_E_CUDA: c_int = -5;
pub const RG_E_NOMEM: c_int = -6;
pub const RG_E_CANCELLED: c_int = -7; // closed channel, rendering.rs:53-54,67
pub const RG_E_LIGHTS: c_int = -8; // obsolete: no longer returned
pub const RG_E_BUSY: c_int = -9;
pub const RG_DEVICE_ALL: i32 = -1;

pub const RG_BODY_SPHERE: u8 = 0;
pub const RG_BODY_PLANE: u8 = 1;
pub const RG_BODY_DISK: u8 = 2;
pub const RG_BODY_AABB: u8 = 3;
pub const RG_COLORATION_COLOR: u8 = 0;
pub const RG_COLORATION_TEXTURE: u8 = 1;
pub const RG_SURFACE_DIFFUSE: u8 = 0;
pub const RG_SURFACE_REFLECTING: u8 = 1;
pub const RG_SURFACE_REFRACTIVE: u8 = 2;
pub const RG_LIGHT_DIRECTIONAL: u8 = 0;
pub const RG_LIGHT_SPHERICAL: u8 = 1;

pub const RG_OPT_PIPELINE: i32 = 1;
pub const RG_OPT_ACCEL: i32 = 2;
pub const RG_OPT_MAX_DEPTH: i32 = 3; // src/main.rs:119-123
pub const RG_OPT_BATCH_PIXELS: i32 = 4;
pub const RG_OPT_VERIFY_CULL: i32 = 5;
pub const RG_OPT_OVERLAP: i32 = 6;
pub const RG_OPT_HOST_FREE: i32 = 7; // obsolete: accepted (0-2) and ignored
pub const RG_OPT_GRAPH: i32 = 8;
pub const RG_OPT_TRACE_STATS: i32 = 9;
pub const RG_OPT_SCHEDULE: i32 = 11;
pub const RG_OPT_TILE_ROWS: i32 = 12;
pub const RG_OPT_ORIGIN_HINTS: i32 = 13;
pub const RG_OPT_SUPERSAMPLE: i32 = 14; // n x n primary rays per pixel (1-8), box-filtered on the device

#[repr(C)]
pub struct rg_texture_desc {
    pub width: u32,
    pub height: u32,
    pub channels: u32,
    pub reserved: u32,
    pub pixels: *const u8,
}

#[repr(C)]
pub struct rg_scene_desc {
    pub abi_version: u32,
    pub max_recursion_depth: u32,
    pub fov: f64,
    pub default_color: [f32; 3],
    pub n_bodies: u32,
    pub body_kind: *const u8,
    pub body_geom: *const f64,
    pub coloration_kind: *const u8,
    pub color: *const f32,
    pub texture_id: *const i32,
    pub texture_offset: *const f32,
    pub albedo: *const f32,
    pub surface_kind: *const u8,
    pub surface_param: *const f32,
    pub n_lights: u32,
    pub n_textures: u32,
    pub light_kind: *const u8,
    pub light_vec: *const f64,
    pub light_color: *const f32,
    pub light_intensity: *const f32,
    pub textures: *const rg_texture_desc,
}

#[repr(C)]
#[derive(Default, Debug, Clone, Copy)]
pub struct rg_stats {
    pub rays_primary: u64,
    pub rays_shadow: u64,
    pub rays_reflection: u64,
    pub rays_transmission: u64,
    pub body_tests: u64,
    pub exact_tests: u64,
    pub cull_unsound: u64,
    pub err_nan_distance: u64,
    pub err_transmission_none: u64,
    pub err_aabb_normal: u64,
    pub ms_device: f64,
    pub ms_trace: f64,
    pub ms_wall: f64,
    pub gpu_launches: u32,
    pub batches: u32,
    pub max_level: u32,
    pub accel_used: u32,
    pub host_free: u32,
    pub graph_replays: u32,
    pub grid_cells: u64,
    pub grid_fetches: u64,
    pub grid_culls: u64,
    pub grid_refills: u64,
    pub grid_lane_steps: u64,
    pub grid_lane_slots: u64,
    pub pipeline_used: u32,
    pub devices_used: u32,
}

pub enum rg_scene {}

pub type rg_rows_cb =
    extern "C" fn(y0: u32, rows: u32, width: u32, rgba: *const u8, user: *mut c_void) -> c_int;

pub type rg_rows_f32_cb =
    extern "C" fn(y0: u32, rows: u32, width: u32, rgb: *const f32, user: *mut c_void) -> c_int;

extern "C" {
    pub fn rg_scene_create(desc: *const rg_scene_desc, device: i32, out: *mut *mut rg_scene) -> c_int;
    pub fn rg_scene_create_multi(desc: *const rg_scene_desc, devices: *const i32, n_devices: u32,
                                 out: *mut *mut rg_scene) -> c_int;
    pub fn rg_scene_device_count(scene: *const rg_scene) -> c_int;
    pub fn rg_scene_destroy(scene: *mut rg_scene);
    pub fn rg_scene_set_option(scene: *mut rg_scene, key: i32, value: i64) -> c_int;
    pub fn rg_render(scene: *mut rg_scene, width: u32, height: u32, rgba_out: *mut u8,
                     stats: *mut rg_stats) -> c_int;
    pub fn rg_render_rows(scene: *mut rg_scene, width: u32, height: u32, y0: u32, y1: u32,
                          rgba_out: *mut u8, stats: *mut rg_stats) -> c_int;
    pub fn rg_render_rows_device(scene: *mut rg_scene, width: u32, height: u32, y0: u32, y1: u32,
                                 d_rgba_out: *mut c_void, cuda_stream: *mut c_void,
                                 stats: *mut rg_stats) -> c_int;
    pub fn rg_render_rowlist_device(scene: *mut rg_scene, width: u32, height: u32, rows: *const u32,
                                    n_rows: u32, d_rgba_out: *mut c_void, cuda_stream: *mut c_void,
                                    stats: *mut rg_stats) -> c_int;
    pub fn rg_render_rowlist_scatter(scene: *mut rg_scene, width: u32, height: u32, rows: *const u32,
                                     n_rows: u32, d_frame: *mut c_void, cuda_stream: *mut c_void,
                                     stats: *mut rg_stats) -> c_int;
    pub fn rg_render_rowlist_host(scene: *mut rg_scene, width: u32, height: u32, rows: *const u32, n_rows: u32,
                                  frame: *mut u8, stats: *mut rg_stats) -> c_int;
    pub fn rg_host_register(ptr: *mut c_void, bytes: usize) -> c_int;
    pub fn rg_host_unregister(ptr: *mut c_void) -> c_int;
    pub fn rg_device_enable_peer(device: i32, peer: i32) -> c_int;
    pub fn rg_shm_barrier_open(name: *const c_char, parties: u32, create: i32, handle: *mut *mut c_void) -> c_int;
    pub fn rg_shm_barrier_wait(handle: *mut c_void) -> c_int;
    pub fn rg_shm_barrier_close(handle: *mut c_void) -> c_int;
    pub fn rg_shared_frame_create(device: i32, bytes: usize, d_ptr: *mut *mut c_void, handle: *mut u8) -> c_int;
    pub fn rg_shared_frame_open(device: i32, handle: *const u8, d_ptr: *mut *mut c_void) -> c_int;
    pub fn rg_shared_frame_close(device: i32, d_ptr: *mut c_void, is_owner: i32) -> c_int;
    pub fn rg_render_stream(scene: *mut rg_scene, width: u32, height: u32, band_rows: u32,
                            cb: rg_rows_cb, user: *mut c_void, stats: *mut rg_stats) -> c_int;
    pub fn rg_render_rows_f32(scene: *mut rg_scene, width: u32, height: u32, y0: u32, y1: u32,
                              rgb_out: *mut f32, stats: *mut rg_stats) -> c_int;
    pub fn rg_render_stream_f32(scene: *mut rg_scene, width: u32, height: u32, band_rows: u32,
                                cb: rg_rows_f32_cb, user: *mut c_void, stats: *mut rg_stats) -> c_int;
    pub fn rg_trim() -> c_int;
    pub fn rg_last_error() -> *const c_char;
    pub fn rg_measure_peaks(device: i32, fp32_tflops: *mut f64, fp64_tflops: *mut f64,
                            sm_clock_mhz: *mut f64) -> c_int;
    pub fn rg_device_count() -> c_int;
}
