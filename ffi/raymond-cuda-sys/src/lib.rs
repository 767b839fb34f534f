// raymond-cuda-sys/src/lib.rs — 1:1 with include/raymond.h, RM_ABI_VERSION 2 (never compiled here: no rustc in the build image)
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] #[derive(Clone, Copy)] pub struct rm_vec3 { pub x: f64, pub y: f64, pub z: f64 }
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_vec2 { pub x: f64, pub y: f64 }
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_ray { pub origin: rm_vec3, pub direction: rm_vec3 }
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_vertex { pub position: rm_vec3, pub normal: rm_vec3, pub uv: rm_vec2, pub tangent: rm_vec3 }
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_triangle { pub v0: rm_vertex, pub v1: rm_vertex, pub v2: rm_vertex }   // == core::geometry::Triangle (264 B)
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_material { pub kind: u32, pub reserved: u32, pub a: rm_vec3, pub b: rm_vec3, pub p0: f64, pub p1: f64 }
/// With `aperture_radius > 0` (depth of field), creating a renderer or task returns RM_ERR_INVALID_ARGUMENT unless
/// `aperture_radius <= 1e150`, `position` is finite and `focal_length >= 0` (not NaN).
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_camera_settings {
    pub backbuffer_width: usize, pub backbuffer_height: usize, pub fov_vert: f64, pub position: rm_vec3,
    pub focal_length: f64, pub aperture_radius: f64 }
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_settings {
    pub worker_count: usize, pub camera_settings: rm_camera_settings, pub sample_count: usize,
    pub samples_per_iteration: usize, pub tile_size: [usize; 2], pub bounce_limit: usize }
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_gpu_options {
    pub device: i32, pub rank: i32, pub world_size: i32, pub partition: u32, pub seed: u64,
    pub stream: *mut c_void, pub accum_device: *mut c_void, pub batch_spp: usize, pub flags: u32, pub device_count: u32,
    pub device_list: *const i32, pub precision: u32, pub reserved: u32 }
#[repr(C)] pub struct rm_tile { pub sample_count: usize, pub width: usize, pub height: usize, pub left: usize, pub top: usize, pub data: *mut rm_vec3 }
#[repr(C)] pub struct rm_message { pub kind: u32, pub reserved: u32, pub tile: rm_tile }
#[repr(C)] #[derive(Default)] pub struct rm_stats {
    pub samples: u64, pub rays: u64, pub nonfinite_samples: u64, pub kernel_launches: u64,
    pub device_ms: f64, pub upload_ms: f64, pub upload_bytes: u64 }
pub enum rm_mesh {} pub enum rm_grid {} pub enum rm_scene {} pub enum rm_task {}

extern "C" {
    pub fn rm_last_error() -> *const c_char;
    pub fn rm_last_status() -> c_int;
    pub fn rm_mesh_from_triangles(t: *const rm_triangle, n: usize) -> *mut rm_mesh;      // Mesh::new          mesh.rs:16
    pub fn rm_mesh_load_ply(path: *const c_char) -> *mut rm_mesh;                        // Mesh::load_ply     mesh.rs:58
    pub fn rm_mesh_translate(m: *mut rm_mesh, t: rm_vec3) -> c_int;                      // bake_transform     mesh.rs:48
    pub fn rm_mesh_destroy(m: *mut rm_mesh);
    pub fn rm_grid_build(m: *mut rm_mesh, status: *mut c_int) -> *mut rm_grid;           // build_from_mesh    acc_grid.rs:36
    pub fn rm_grid_retain(g: *mut rm_grid) -> *mut rm_grid;                              // Arc::clone
    pub fn rm_grid_release(g: *mut rm_grid);                                             // drop
    pub fn rm_scene_create() -> *mut rm_scene;                                           // Scene::new         scene.rs:48
    pub fn rm_scene_add_sphere(s: *mut rm_scene, o: rm_vec3, r: f64, m: *const rm_material) -> c_int;
    pub fn rm_scene_add_plane(s: *mut rm_scene, o: rm_vec3, n: rm_vec3, m: *const rm_material) -> c_int;
    pub fn rm_scene_add_grid(s: *mut rm_scene, g: *mut rm_grid, m: *const rm_material) -> c_int;
    pub fn rm_scene_destroy(s: *mut rm_scene);
    pub fn rm_scene_intersect(s: *const rm_scene, device: c_int, rays: *const rm_ray, n: usize,
                              obj: *mut i64, sub: *mut u64, dist: *mut f64) -> c_int;     // Scene::intersect   scene.rs:54
    pub fn rm_render_tiled(s: *const rm_scene, st: *const rm_settings, o: *const rm_gpu_options) -> *mut rm_task; // trace.rs:137
    pub fn rm_task_poll(t: *mut rm_task, out: *mut rm_message) -> c_int;                 // TaskHandle::poll   trace.rs:115
    pub fn rm_task_await(t: *mut rm_task, out: *mut rm_vec3) -> c_int;                   // TaskHandle::await  trace.rs:82
    pub fn rm_task_set_callback(t: *mut rm_task, cb: Option<extern "C" fn(*const rm_tile, *mut c_void)>, user: *mut c_void) -> c_int;
    pub fn rm_task_pump(t: *mut rm_task) -> c_int;                                       // async_await        trace.rs:119
    pub fn rm_task_finished(t: *mut rm_task) -> c_int;
    pub fn rm_task_stats(t: *mut rm_task, out: *mut rm_stats) -> c_int;
    pub fn rm_task_destroy(t: *mut rm_task);
    pub fn rm_tile_free(t: *mut rm_tile);
}

// ---- entry points added after the first draft of INTEGRATION.md (include/raymond.h)
extern "C" {
    pub fn rm_grid_build_on_device(m: *mut rm_mesh, device: c_int, status: *mut c_int) -> *mut rm_grid;   // build_from_mesh, cell lists built on the GPU
    pub fn rm_project_load_scene(path: *const c_char, status: *mut c_int) -> *mut rm_scene;                // Project::load + build_scene  project.rs:33-57
    pub fn rm_message_to_json(m: *const rm_message, buf: *mut c_char, cap: usize) -> usize;                // protocol.rs:9-14
    pub fn rm_tonemap_rgb8(frame: *const rm_vec3, pixels: usize, exposure: f64, gamma: f64, device: c_int, out: *mut u8) -> c_int; // cli_old main.rs:157-181
    pub fn rm_write_png(path: *const c_char, rgb8: *const u8, width: usize, height: usize) -> c_int;       // cli_old main.rs:194-197
    pub fn rm_release_cached_memory() -> c_int;
    pub fn rm_measure_fp64_rate(device: c_int, gops_out: *mut f64) -> c_int;                                // diagnostic (roofline)
}

// ---- per-tile adaptive sampling (include/raymond.h).  E_t of a tile after n >= 2 samples, per pixel and channel from the
// running sum S and the running sum of squares Q: m = S/n, v = max(Q - S*m, 0)/(n-1), se2 = v/n;
// r_p = sqrt(se2_R + se2_G + se2_B) / (m_R + m_G + m_B + 1e-3); E_t = sqrt(mean over the tile of r_p^2); converged iff E_t <= threshold.
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_adaptive_settings { pub threshold: f64, pub min_samples: usize }
pub enum rm_renderer {}
extern "C" {
    // render_tiled with TileFinished(n) for every tile that converged at checkpoint n; NULL settings = rm_render_tiled.
    // rm_task_pump still stops at the first message that is not TileProgressed: read an adaptive task with poll / await.
    pub fn rm_render_tiled_adaptive(s: *const rm_scene, st: *const rm_settings, o: *const rm_gpu_options,
                                    a: *const rm_adaptive_settings) -> *mut rm_task;
    pub fn rm_renderer_read_moments(r: *mut rm_renderer, out: *mut rm_vec3) -> c_int;
    pub fn rm_renderer_tile_errors(r: *mut rm_renderer, sample_count: usize, out: *mut f64, capacity: usize) -> usize;
    pub fn rm_renderer_set_active_tiles(r: *mut rm_renderer, active: *const u8, tile_count: usize) -> c_int;
}

// ---- first-hit feature buffers (RM_FLAG_AOV) and the feature-guided a-trous denoiser (include/raymond.h states the filter).
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_denoise_settings {
    pub iterations: u32,   // 1..10
    pub reserved: u32,
    pub sigma_color: f64, pub sigma_normal: f64, pub sigma_albedo: f64, pub sigma_depth: f64,   // finite, > 0
}
extern "C" {
    // feature sums / sample_count, W*H each; any output may be null; RM_ERR_STATE without RM_FLAG_AOV
    pub fn rm_renderer_read_aovs(r: *mut rm_renderer, sample_count: usize, albedo: *mut rm_vec3, normal: *mut rm_vec3, depth: *mut f64) -> c_int;
    // null settings = the defaults; needs RM_FLAG_AOV | RM_FLAG_MOMENTS, sample_count >= 2 and a renderer with world_size <= 1
    pub fn rm_renderer_read_denoised(r: *mut rm_renderer, sample_count: usize, settings: *const rm_denoise_settings, out: *mut rm_vec3) -> c_int;
    // render_tiled that also filters the finished frame across the task's devices; messages and rm_task_await are rm_render_tiled's.
    // null settings = the defaults; sample_count >= 2; not for one rank of a multi-process job
    pub fn rm_render_tiled_denoised(s: *const rm_scene, st: *const rm_settings, o: *const rm_gpu_options,
                                    d: *const rm_denoise_settings) -> *mut rm_task;
    // blocks until the task is finished, then the W*H filtered frame; RM_ERR_STATE for a task not made by rm_render_tiled_denoised
    pub fn rm_task_await_denoised(t: *mut rm_task, out: *mut rm_vec3) -> c_int;
}

// ---- environment maps (include/raymond.h states the lookup and what a ray that leaves the scene delivers)
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_environment {
    pub texels: *const f32,            // width*height RGB triples, row-major, row 0 = +y; copied
    pub width: usize, pub height: usize, // 1..32768 each
    pub scale: f64,                    // finite, >= 0
    pub rotation: f64,                 // radians about +y, finite
}
extern "C" {
    // null env clears the map; RM_ERR_INVALID_ARGUMENT (scene unchanged) for a NaN / Inf / negative texel or a bad size, scale or rotation
    pub fn rm_scene_set_environment(s: *mut rm_scene, env: *const rm_environment) -> c_int;
    // Radiance RGBE (.hdr); texels null = only the size; RM_ERR_IO / RM_ERR_IMAGE
    pub fn rm_load_hdr(path: *const c_char, width: *mut usize, height: *mut usize, texels: *mut f32) -> c_int;
}
pub const RM_ERR_IMAGE: c_int = -12;            // a malformed or unsupported image file (rm_load_hdr)

// ---- colour textures (include/raymond.h states the uv of each geometry kind, the lookup and what a textured colour replaces)
#[repr(C)] #[derive(Clone, Copy)] pub struct rm_texture {
    pub texels: *const f32,            // width*height RGB triples, row-major, row 0 = top; copied
    pub width: usize, pub height: usize, // 1..32768 each
    pub scale_u: f64, pub scale_v: f64, // finite
}
extern "C" {
    // null texture unbinds; RM_ERR_INVALID_ARGUMENT (scene unchanged) for a bad index, a NaN / Inf / negative texel, a bad size
    // or scale; RM_ERR_UNSUPPORTED for an Emission object
    pub fn rm_scene_set_texture(s: *mut rm_scene, object_index: usize, texture: *const rm_texture) -> c_int;
}

// ---- values of the enum / flag fields (include/raymond.h, RM_ABI_VERSION 2)
pub const RM_PARTITION_SAMPLES: u32 = 0;        // rank g renders global samples g, g+G, ...
pub const RM_PARTITION_TILES: u32 = 1;          // tiles dealt round-robin in the reference's queue order (src/trace.rs:146-172)
pub const RM_PRECISION_F64: u32 = 0;            // the reference's f64 arithmetic throughout
pub const RM_PRECISION_F32_SHADING: u32 = 1;    // BRDF sampling / weights in f32; intersections, hit points, normals stay f64
pub const RM_FLAG_KEEP_NONFINITE: u32 = 1;
pub const RM_FLAG_STAGE_TIMING: u32 = 2;
pub const RM_FLAG_COUNT_WORK: u32 = 4;
pub const RM_FLAG_MOMENTS: u32 = 64;            // keep the running sums of squared samples (rm_renderer_read_moments / tile_errors)
pub const RM_FLAG_AOV: u32 = 128;               // keep the first-hit albedo / normal / depth sums (rm_renderer_read_aovs / read_denoised)
pub const RM_TILE_FINISHED: u32 = 0;            // Message::TileFinished
pub const RM_TILE_PROGRESSED: u32 = 1;          // Message::TileProgressed
