/*
 * raymond.h — C ABI of the B200-native path-tracing hot path.
 *
 * This header is the drop-in boundary: every type and entry point below is the
 * C image of one item of the reference's Rust API (Nyrox/raymond) for the
 * per-pixel Monte-Carlo path-tracing path, and names the reference interface it
 * replaces as `file:line` relative to the reference checkout.  A maintainer of
 * the reference binds these with a thin `extern "C"` FFI crate (see
 * INTEGRATION.md); nothing here exposes a torch or CUDA runtime type.
 *
 * Conventions
 *   - all arithmetic types are the reference's: f64 (`TFloat = f64`,
 *     core/src/math.rs:10) and usize (size_t);
 *   - functions returning `int` return RM_OK (0) or a negative rm_status; they
 *     never unwind across the boundary.  The reference panics instead
 *     (unwrap/expect/panic! — src/trace.rs:212,218,253; acc_grid.rs:47,51,61);
 *     each panic site maps to a status below.  rm_last_error() returns a
 *     thread-local description of the last failure on the calling thread;
 *   - objects are reference counted where the reference uses Arc
 *     (core/src/scene.rs:12) and are snapshotted where the reference takes
 *     arguments by value (src/trace.rs:137);
 *   - there is no CPU implementation behind this ABI: every compute entry point
 *     runs CUDA kernels built for sm_100a and fails with RM_ERR_CUDA when no
 *     device is usable.
 */
#ifndef RAYMOND_H
#define RAYMOND_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RM_ABI_VERSION 2

/* ------------------------------------------------------------------ status */

typedef enum rm_status {
    RM_OK = 0,
    RM_ERR_INVALID_ARGUMENT = -1,
    RM_ERR_IO = -2,               /* fs::read_to_string(..).unwrap()           mesh.rs:59      */
    RM_ERR_PLY = -3,              /* parse::<f64>().unwrap(), values[..] OOB   mesh.rs:69-113  */
    RM_ERR_GRID_INDEX_OOB = -4,   /* naive_cells[..] index out of bounds       acc_grid.rs:61  */
    RM_ERR_DEGENERATE_BOUNDS = -5,/* res 0 => `grid_res[i] - 1` underflow      acc_grid.rs:54  */
    RM_ERR_GRID_CAST = -6,        /* expect("Failed to cast cell bounds ..")   acc_grid.rs:47,51 */
    RM_ERR_CUDA = -7,
    RM_ERR_UNSUPPORTED = -8,
    RM_ERR_OUT_OF_MEMORY = -9,
    RM_ERR_STATE = -10,
    RM_ERR_PROJECT = -11          /* serde_json::from_reader(file)? fails     project.rs:35   */
} rm_status;

const char* rm_last_error(void);
/* rm_status of the last failure on the calling thread — for the entry points that return a handle (NULL on failure). */
int rm_last_status(void);
int rm_abi_version(void);

/* ------------------------------------------------------------- plain types */

/* cgmath::Vector3<f64> / Vector2<f64>           core/src/lib.rs:5-6 */
typedef struct rm_vec3 { double x, y, z; } rm_vec3;
typedef struct rm_vec2 { double x, y; } rm_vec2;

/* Ray { origin, direction }                     core/src/geometry/mod.rs:37-41 */
typedef struct rm_ray { rm_vec3 origin; rm_vec3 direction; } rm_ray;

/* Vertex { position, normal, uv, tangent }      core/src/geometry/primitives/vertex.rs:5-10 */
typedef struct rm_vertex {
    rm_vec3 position;
    rm_vec3 normal;
    rm_vec2 uv;
    rm_vec3 tangent;
} rm_vertex;

/* Triangle(Vertex, Vertex, Vertex)              core/src/geometry/primitives/triangle.rs:8
 * 3 x 88 B = 264 B, same field order as the reference. */
typedef struct rm_triangle { rm_vertex v0, v1, v2; } rm_triangle;

/* AABB { min, max }                             core/src/geometry/primitives/aabb.rs:4-7 */
typedef struct rm_aabb { rm_vec3 min; rm_vec3 max; } rm_aabb;

/* enum Material { Diffuse(Vector3, f64), Metal(Vector3, f64),
 *                 Emission(Vector3, Vector3, f64, f64) }          core/src/lib.rs:21-26
 *   Diffuse : a = colour, p0 = roughness
 *   Metal   : a = colour, p0 = roughness
 *   Emission: a = emitted radiance, b / p0 / p1 = the three fields the
 *             integrator ignores (src/trace.rs:250) — kept so a scene
 *             round-trips. */
typedef enum rm_material_kind {
    RM_MATERIAL_DIFFUSE = 0,
    RM_MATERIAL_METAL = 1,
    RM_MATERIAL_EMISSION = 2
} rm_material_kind;

typedef struct rm_material {
    uint32_t kind;   /* rm_material_kind */
    uint32_t reserved;
    rm_vec3 a;
    rm_vec3 b;
    double p0;
    double p1;
} rm_material;

/* ------------------------------------------------------- mesh, grid, scene */

typedef struct rm_mesh rm_mesh;     /* Mesh { triangles, bounding_box }  core/src/geometry/mesh.rs:10-13 */
typedef struct rm_grid rm_grid;     /* Arc<AccGrid>                      core/src/geometry/acc_grid.rs:27-33 */
typedef struct rm_scene rm_scene;   /* Scene { objects }                 core/src/scene.rs:42-45 */

/* Mesh::new(Vec<Triangle>)                      mesh.rs:16-21 (copies the triangles, computes the bounds) */
rm_mesh* rm_mesh_from_triangles(const rm_triangle* triangles, size_t count);
/* Mesh::load_ply(PathBuf)                       mesh.rs:58-121 (ASCII PLY, x y z nx ny nz [s t], triangles only) */
rm_mesh* rm_mesh_load_ply(const char* path);
/* Mesh::bake_transform(translate)               mesh.rs:48-56 */
int rm_mesh_translate(rm_mesh* mesh, rm_vec3 translate);
size_t rm_mesh_triangle_count(const rm_mesh* mesh);
int rm_mesh_bounds(const rm_mesh* mesh, rm_aabb* out);
/* read back triangles [first, first+count) */
int rm_mesh_triangles(const rm_mesh* mesh, size_t first, size_t count, rm_triangle* out);
void rm_mesh_destroy(rm_mesh* mesh);

/* AccGrid::build_from_mesh(mesh)                acc_grid.rs:36-83.  Like the Rust
 * move, the grid takes the triangles out of `mesh`; the (now empty) mesh handle
 * must still be destroyed by the caller.  Returns NULL on failure with
 * rm_last_error() set; `*status` (optional) receives the rm_status. */
rm_grid* rm_grid_build(rm_mesh* mesh, int* status);
/* The same AccGrid::build_from_mesh with the cell lists counted, scanned and filled by CUDA kernels on `device`
 * (identical resolution, cell size and per-cell triangle lists, in the same ascending order, and the same failure
 * statuses as rm_grid_build).  For meshes of millions of triangles, where the host build takes seconds. */
rm_grid* rm_grid_build_on_device(rm_mesh* mesh, int device, int* status);
rm_grid* rm_grid_retain(rm_grid* grid);   /* Arc::clone */
void rm_grid_release(rm_grid* grid);      /* drop */

typedef struct rm_grid_info {
    size_t resolution[3];      /* AccGrid.resolution                 acc_grid.rs:31 */
    rm_vec3 cell_size;         /* AccGrid.cell_size                  acc_grid.rs:32 */
    rm_aabb bounds;            /* mesh.bounding_box                                 */
    size_t cell_count;         /* cells.len()                                       */
    size_t reference_count;    /* mapping_table.len() - cells.len()                 */
    size_t triangle_count;
} rm_grid_info;
int rm_grid_get_info(const rm_grid* grid, rm_grid_info* out);
/* The grid in compressed-row form: `cell_start` has cell_count+1 entries,
 * `references` has reference_count entries; the references of cell c are
 * references[cell_start[c] .. cell_start[c+1]) in ascending triangle order —
 * the same contents and order as mapping_table[cells[c]+1 ..] (acc_grid.rs:67-74). */
int rm_grid_get_cells(const rm_grid* grid, uint32_t* cell_start, uint32_t* references);

/* Scene::new()                                  scene.rs:48-52 */
rm_scene* rm_scene_create(void);
/* scene.objects.push(Object { geometry: Geometry::Sphere(Sphere{origin, radius}), material })
 *                                               scene.rs:9-13,33-37; sphere.rs:5-8 */
int rm_scene_add_sphere(rm_scene* scene, rm_vec3 origin, double radius, const rm_material* material);
/* Geometry::Plane(Plane{origin, normal})        plane.rs:5-8 */
int rm_scene_add_plane(rm_scene* scene, rm_vec3 origin, rm_vec3 normal, const rm_material* material);
/* Geometry::Grid(Arc<AccGrid>) — retains the grid   scene.rs:12 */
int rm_scene_add_grid(rm_scene* scene, rm_grid* grid, const rm_material* material);
/* Project::load(path)?.build_scene()             core/src/project.rs:33-57.  The serde_json project file
 * ({"objects":[{"geometry":{"Sphere"|"Plane"|"Mesh": ..},"material":{"Diffuse"|"Metal"|"Emission": [..]}}]}, externally
 * tagged enums, cgmath vectors as {"x","y","z"}); a Mesh path is loaded with Mesh::load_ply and built into a grid. */
rm_scene* rm_project_load_scene(const char* path, int* status);
size_t rm_scene_object_count(const rm_scene* scene);
void rm_scene_destroy(rm_scene* scene);

/* Scene::intersect(&self, Ray) -> Option<(&Object, Hit)>          scene.rs:54-74
 * batched over `count` rays held in HOST memory; results to HOST memory:
 *   object_index[i]    index into scene.objects, -1 for a miss
 *   subobject_index[i] Hit.subobject_index (triangle index for a grid, else 0)
 *   distance[i]        Hit.distance (untouched on a miss)
 * Bit-exact with the reference's f64 decision sequence (no FMA contraction).
 * Any output pointer may be NULL.  `device` is the CUDA ordinal to run on. */
int rm_scene_intersect(const rm_scene* scene, int device, const rm_ray* rays, size_t count,
                       int64_t* object_index, uint64_t* subobject_index, double* distance);

/* --------------------------------------------------------------- settings */

/* CameraSettings                                src/trace.rs:32-40
 * `position` is `transform.position` (Transform is position-only, src/transform.rs:4-6).
 * With aperture_radius > 0 (depth of field), rm_renderer_create*, rm_render_tiled and rm_render_tiled_adaptive return
 * RM_ERR_INVALID_ARGUMENT, before any device work, unless aperture_radius <= 1e150, position is finite and
 * focal_length >= 0 (not NaN): otherwise the reference's aperture sampling never ends, or its focal-plane unwrap panics. */
typedef struct rm_camera_settings {
    size_t backbuffer_width;
    size_t backbuffer_height;
    double fov_vert;          /* degrees */
    rm_vec3 position;
    double focal_length;
    double aperture_radius;   /* > 0 selects generate_primary_ray_with_dof (src/trace.rs:335-360) */
} rm_camera_settings;

/* Settings                                      src/trace.rs:42-55 */
typedef struct rm_settings {
    size_t worker_count;            /* CPU threads in the reference; ignored by the GPU path */
    rm_camera_settings camera_settings;
    size_t sample_count;
    size_t samples_per_iteration;   /* 0: only TileFinished messages */
    size_t tile_size[2];            /* (width, height) */
    size_t bounce_limit;
} rm_settings;

typedef enum rm_partition {
    RM_PARTITION_SAMPLES = 0,   /* rank g renders global samples g, g+G, g+2G, ... of every pixel */
    RM_PARTITION_TILES = 1      /* tiles dealt round-robin in the reference's tile order (src/trace.rs:146-172) */
} rm_partition;

/* Arithmetic of the STATISTICAL scope (BRDF sampling and weights, src/trace.rs:256-319,362-416).  The bit-exact scope —
 * camera rays, Scene::intersect, hit points, normals, ray offsets — is always the reference's f64 sequence. */
typedef enum rm_precision {
    RM_PRECISION_F64 = 0,       /* every operation is the reference's f64 operation, in its order (same-stream parity with the oracle) */
    RM_PRECISION_F32_SHADING = 1 /* lobe sampling, Fresnel, GGX and Smith terms in f32 with FMA; agrees with the f64 mode within Monte-Carlo noise */
} rm_precision;

/* Non-finite samples.  By default a sample whose value is NaN / Inf is dropped and counted (rm_stats.nonfinite_samples), and a
 * path whose throughput became exactly (0,0,0) is stopped early.  With RM_FLAG_KEEP_NONFINITE every path is traced the way the
 * reference traces it — no early stop; a path that ends without emission delivers throughput (*) 0, and at the bounce limit
 * throughput (*) last weight (*) 0 — and every sample is accumulated, so a NaN / Inf weight anywhere on a path poisons its
 * pixel exactly where the reference's does, and nonfinite_samples equals the reference's count. */
#define RM_FLAG_KEEP_NONFINITE 1u
#define RM_FLAG_STAGE_TIMING 2u    /* bracket every kernel launch with CUDA events; totals per wavefront stage in rm_stage_stats */
#define RM_FLAG_COUNT_WORK 4u      /* instrumented kernels: count grid cells visited and triangle tests per stage (slower) */
#define RM_FLAG_NO_RAY_BINNING 8u  /* reserved: accepted, no effect (the bounced rays are always traversed in queue order) */
#define RM_FLAG_FUSE_SETUP 16u     /* reserved: accepted, no effect (shading and the next depth's set-up are separate kernels) */
#define RM_FLAG_SPLIT_SETUP 32u    /* reserved: accepted, no effect (shading and the next depth's set-up are separate kernels) */
/* Second moments: next to the running sum S the renderer keeps, per pixel and channel, the running sum of squared sample
 * values Q, under the same rule as S — samples added in global sample order; non-finite samples left out of both by default,
 * added to both with RM_FLAG_KEEP_NONFINITE.  Read with rm_renderer_read_moments; used by rm_renderer_tile_errors. */
#define RM_FLAG_MOMENTS 64u

/* GPU-side knobs that have no counterpart in the reference. Zero-initialise
 * for defaults (device 0, one rank, library-owned stream and buffers). */
typedef struct rm_gpu_options {
    int32_t device;          /* CUDA ordinal */
    int32_t rank;            /* this process's share: rank of world_size */
    int32_t world_size;      /* 0 or 1 = everything */
    uint32_t partition;      /* rm_partition */
    uint64_t seed;           /* key of the counter-based RNG */
    void* stream;            /* cudaStream_t to launch on; NULL = a stream the library creates */
    void* accum_device;      /* optional caller-owned device buffer, W*H rm_vec3 (f64 sums), zeroed by the library */
    size_t batch_spp;        /* samples per pixel per wavefront batch; 0 = auto */
    uint32_t flags;          /* RM_FLAG_* */
    uint32_t device_count;   /* rm_render_tiled only: > 1 renders on `device_count` devices from THIS process (one stream per
                              * device, `partition` between them); the accumulators are combined over NVLink (every device sums
                              * its slice of the frame from all peers, in device order) straight into the frame the caller reads.
                              * rank / world_size are then set by the library.  0 or 1 = one GPU. */
    const int32_t* device_list; /* the `device_count` CUDA ordinals to use; NULL = device, device+1, ...  An ordinal may appear more
                              * than once (several shares of the frame rendered on one GPU: same data path — scene placement, peer
                              * reduce, progressive tiles — on a box with fewer GPUs). */
    uint32_t precision;      /* rm_precision */
    uint32_t reserved;
} rm_gpu_options;

/* Tile { sample_count, width, height, left, top, data }   core/src/tile.rs:6-14
 * `data` is the RUNNING SUM of radiance (not the mean), row-major inside the tile. */
typedef struct rm_tile {
    size_t sample_count;
    size_t width;
    size_t height;
    size_t left;
    size_t top;
    rm_vec3* data;   /* width*height entries; owned by the receiver — rm_tile_free */
} rm_tile;
void rm_tile_free(rm_tile* tile);

/* enum Message { TileFinished(Tile), TileProgressed(Tile) }   src/trace.rs:62-66 */
typedef enum rm_message_kind { RM_TILE_FINISHED = 0, RM_TILE_PROGRESSED = 1 } rm_message_kind;
typedef struct rm_message { uint32_t kind; uint32_t reserved; rm_tile tile; } rm_message;

/* The message on the wire (server/src/protocol.rs:9-14: serde tag = "type", content = "data"; Tile per
 * core/src/tile.rs:6-14): {"type":"TileProgressed","data":{"sample_count":..,"width":..,"height":..,"left":..,"top":..,
 * "data":[{"x":..,"y":..,"z":..},..]}}.  Returns the length of the JSON text (without the terminator); writes at most
 * capacity-1 characters + NUL when `buffer` is non-NULL.  Call with NULL to size the buffer. */
size_t rm_message_to_json(const rm_message* message, char* buffer, size_t capacity);

/* ---------------------------------------------------------- render driver */

typedef struct rm_task rm_task;   /* TaskHandle  src/trace.rs:70-75 */

/* render_tiled(scene, settings) -> TaskHandle   src/trace.rs:137-230
 * Returns immediately; the scene and settings are snapshotted (the caller may
 * destroy them).  `options` may be NULL. */
rm_task* rm_render_tiled(const rm_scene* scene, const rm_settings* settings, const rm_gpu_options* options);
/* TaskHandle::poll() -> Option<Message>         src/trace.rs:115-117.  1 = message written, 0 = none. */
int rm_task_poll(rm_task* task, rm_message* out);
/* TaskHandle::r#await() -> Vec<Vector3>         src/trace.rs:82-113.  Blocks until the
 * render is done, then writes W*H averaged pixels (sum / sample_count), row-major.
 * Unlike the reference it skips TileProgressed messages instead of stopping at
 * the first one, and waits on a condition variable instead of a 500 ms sleep. */
int rm_task_await(rm_task* task, rm_vec3* out);
/* set_callback / async_await                    src/trace.rs:78-80,119-134.  The callback
 * runs on the caller's thread from rm_task_pump(), once per pending
 * TileProgressed message; the tile is only valid during the call. */
typedef void (*rm_tile_callback)(const rm_tile* tile, void* user);
int rm_task_set_callback(rm_task* task, rm_tile_callback callback, void* user);
int rm_task_pump(rm_task* task);
/* alive_thread_count == 0                       src/trace.rs:74,89 */
int rm_task_finished(rm_task* task);

typedef struct rm_stats {
    uint64_t samples;            /* paths started */
    uint64_t rays;               /* Scene::intersect evaluations */
    uint64_t nonfinite_samples;  /* samples with a NaN / Inf channel.  With RM_FLAG_KEEP_NONFINITE: kept, and the reference's count.
                                  * Without it: dropped, and counted as this library's paths produce them — a lower bound of the
                                  * reference's count, since a path stopped at a zero throughput, a miss or the bounce limit
                                  * delivers an exact 0 where the reference's product with a NaN / Inf weight is NaN. */
    uint64_t kernel_launches;    /* launches of this library's kernels */
    double device_ms;            /* CUDA-event time of the render section */
    double upload_ms;            /* host flatten + H2D of the scene */
    uint64_t upload_bytes;       /* bytes copied host -> device for the scene and the pixel map */
} rm_stats;
int rm_task_stats(rm_task* task, rm_stats* out);
void rm_task_destroy(rm_task* task);

/* Per-tile adaptive sampling.  The error estimate of a tile after n >= 2 samples, per pixel p and channel c, from the
 * running sum S and the running sum of squares Q (RM_FLAG_MOMENTS):
 *   m = S / n,   v = max(Q - S * m, 0) / (n - 1),   se2 = v / n,
 *   r_p = sqrt(se2_R + se2_G + se2_B) / (m_R + m_G + m_B + 1e-3),   E_t = sqrt(mean over the tile's pixels of r_p^2).
 * A tile has converged iff E_t <= threshold.  A NaN anywhere makes that comparison false, so a NaN-poisoned tile of
 * RM_FLAG_KEEP_NONFINITE renders to the full count.  Without that flag n still counts the dropped samples, as the mean does. */
typedef struct rm_adaptive_settings {
    double threshold;       /* finite, > 0 */
    size_t min_samples;     /* no tile stops before max(min_samples, 2) samples */
} rm_adaptive_settings;
/* render_tiled with per-tile early stopping.  `adaptive` NULL = exactly rm_render_tiled.  Otherwise, at every progressive
 * checkpoint n (every samples_per_iteration samples) with n >= max(min_samples, 2) and n < sample_count, each tile still
 * rendering with E_t <= threshold gets TileFinished(sample_count = n) and is never rendered again; the others get
 * TileProgressed(n) as in rm_render_tiled.  The messages of one checkpoint are in queue order.  A tile that stops early holds
 * exactly the first n samples of the full render.  rm_task_await divides every tile by its own count; rm_stats.samples
 * counts the paths actually started.  rm_task_pump keeps its reference semantics — it stops at the first message that is
 * not TileProgressed — so read an adaptive task with rm_task_poll or rm_task_await.
 * Checked before any device work: a threshold that is not finite or <= 0 and samples_per_iteration == 0 fail with
 * RM_ERR_INVALID_ARGUMENT; one rank of a multi-process job (world_size > 1 with device_count <= 1) with RM_ERR_UNSUPPORTED. */
rm_task* rm_render_tiled_adaptive(const rm_scene* scene, const rm_settings* settings, const rm_gpu_options* options,
                                  const rm_adaptive_settings* adaptive);

/* -------------------------------------------------- device-level interface
 * The pieces rm_render_tiled is made of, for hosts that own the device memory,
 * the stream and the cross-GPU exchange themselves (one process per GPU with
 * an NCCL reduce of the accumulators between rm_renderer_render and
 * rm_renderer_read_frame). */

typedef struct rm_device_scene rm_device_scene;   /* a Scene flattened and resident in HBM */
rm_device_scene* rm_device_scene_create(const rm_scene* scene, int device);
void rm_device_scene_destroy(rm_device_scene* ds);
/* Scene::intersect on rays and results resident in DEVICE memory (same layout
 * and semantics as rm_scene_intersect); asynchronous on `stream`. */
int rm_device_scene_intersect(rm_device_scene* ds, const rm_ray* rays_device, size_t count,
                              int64_t* object_index_device, uint64_t* subobject_index_device,
                              double* distance_device, void* stream);
/* generate_primary_ray for pixel centres (the jitter term forced to 0) of the
 * whole W x H frame, row-major, into DEVICE memory — the C4 ray set. */
int rm_primary_rays_device(const rm_camera_settings* camera, int device, rm_ray* rays_device, void* stream);

typedef struct rm_renderer rm_renderer;
rm_renderer* rm_renderer_create(const rm_scene* scene, const rm_settings* settings, const rm_gpu_options* options);
rm_renderer* rm_renderer_create_on(rm_device_scene* ds, const rm_settings* settings, const rm_gpu_options* options);
/* Enqueue `count` samples per owned pixel: global sample indices
 * first, first+stride, ...  Asynchronous on the renderer's stream. */
int rm_renderer_render(rm_renderer* r, size_t first_sample, size_t count, size_t stride);
/* Device pointer of the W*H rm_vec3 running sums. */
void* rm_renderer_accum_device(rm_renderer* r);
int rm_renderer_clear(rm_renderer* r);   /* zero the running sums (statistics stay cumulative) */
int rm_renderer_sync(rm_renderer* r);
/* D2H of the running sums (no division). */
int rm_renderer_read_sums(rm_renderer* r, rm_vec3* out_host);
/* D2H of sum / sample_count, row-major W*H. */
int rm_renderer_read_frame(rm_renderer* r, size_t sample_count, rm_vec3* out_host);
/* The display transform of the reference's front-end (cli_old/src/main.rs:157-181) as an epilogue kernel on the
 * accumulator: p = sum / sample_count; 1 - exp(p * -1.0 * exposure); powf(1 / gamma); * 255; cast::<u8>() — a pixel
 * with a NaN / out-of-range channel stays (0, 0, 0).  Writes W*H*3 bytes, row-major RGB, to HOST memory. */
int rm_renderer_read_rgb8(rm_renderer* r, size_t sample_count, double exposure, double gamma, uint8_t* out_host);
/* D2H of the running sums of squared samples Q (RM_FLAG_MOMENTS), row-major W*H; RM_ERR_STATE without the flag. */
int rm_renderer_read_moments(rm_renderer* r, rm_vec3* out_host);
/* E_t (defined above rm_adaptive_settings) of every tile after `sample_count` samples, computed on the device from this renderer's S and
 * Q, in rm_tile_layout order; tiles outside the renderer's share (RM_PARTITION_TILES) are NaN.  Writes min(count, capacity)
 * values and returns the tile count (0 on failure, with rm_last_error set).  Needs RM_FLAG_MOMENTS. */
size_t rm_renderer_tile_errors(rm_renderer* r, size_t sample_count, double* out, size_t capacity);
/* Later rm_renderer_render calls render only the tiles of the renderer's share whose `active` entry (rm_tile_layout order,
 * `tile_count` = the layout's count) is non-zero; the sums of the other tiles are left untouched.  NULL = every tile.
 * Asynchronous on the renderer's stream. */
int rm_renderer_set_active_tiles(rm_renderer* r, const uint8_t* active, size_t tile_count);
int rm_renderer_stats(rm_renderer* r, rm_stats* out);

/* Per-stage breakdown of the wavefront.  Slot d (1 <= d < RM_STAGE_SLOTS) is the stage that traces
 * and shades the rays of depth d (deeper stages share the last slot).  A stage is three kernels —
 * kind 0 set-up (ray generation / analytic objects / grid entry), kind 1 grid traversal, kind 2
 * shading — kind 3, slot 0 is the accumulator kernel; kind 4 is reserved (no kernel of this version is counted
 * there, it stays zero).  `ms` / `launches` need
 * RM_FLAG_STAGE_TIMING; `cells` / `triangle_tests` need RM_FLAG_COUNT_WORK; the rest is always
 * counted.  cells = C and triangle_tests = T of the algorithmic bytes-per-ray model
 * (SURVEY.md §8d: 64 + 8 C + 76 T, + 72 per shaded triangle hit). */
#define RM_STAGE_SLOTS 16
#define RM_KERNEL_KINDS 5
typedef struct rm_stage_stats {
    double ms[RM_KERNEL_KINDS][RM_STAGE_SLOTS];
    uint64_t launches[RM_KERNEL_KINDS][RM_STAGE_SLOTS];
    uint64_t rays[RM_STAGE_SLOTS];            /* Scene::intersect evaluations */
    uint64_t grid_rays[RM_STAGE_SLOTS];       /* of those, rays that entered a grid traversal */
    uint64_t cells[RM_STAGE_SLOTS];
    uint64_t triangle_tests[RM_STAGE_SLOTS];
    uint64_t shaded_triangles[RM_STAGE_SLOTS];
    uint64_t evaluated_tests[RM_STAGE_SLOTS];  /* of triangle_tests, the ones NOT proven misses by the bounding-sphere pre-test (RM_FLAG_COUNT_WORK) */
    uint64_t occupied_cells[RM_STAGE_SLOTS];   /* of cells, the ones with a non-empty list (RM_FLAG_COUNT_WORK) */
    uint64_t evaluated_test_flops[RM_STAGE_SLOTS]; /* f64 add/sub/mul/div executed by the evaluated Triangle::intersects calls: 20, 30, 46 or 52
                                                * per call depending on the exit taken, triangle.rs:11-44 (RM_FLAG_COUNT_WORK) */
} rm_stage_stats;
int rm_renderer_stage_stats(rm_renderer* r, rm_stage_stats* out);
void rm_renderer_destroy(rm_renderer* r);

/* The same display transform for an averaged frame held in HOST memory (what rm_task_await returns). */
int rm_tonemap_rgb8(const rm_vec3* frame_host, size_t pixels, double exposure, double gamma, int device, uint8_t* out_host);
/* image.save("output.png")                      cli_old/src/main.rs:194-197: 8-bit RGB PNG (host code). */
int rm_write_png(const char* path, const uint8_t* rgb8, size_t width, size_t height);

/* Diagnostic for the roofline (SURVEY 8d): the f64 operation rate this device sustains on a stream of independent DADD / DMUL
 * (no FMA, as this library is compiled), in Gop/s.  Runs a ~10 ms kernel on `device`. */
int rm_measure_fp64_rate(int device, double* gops_out);

/* The library keeps what the next frame of the same job needs again: the wavefront queues (a private stream-ordered pool per
 * GPU, up to 48 GiB cached), scene blocks and accumulators (up to 16 GiB), the pixel launch order per frame layout (up to
 * 512 MiB) and pinned staging blocks.  This returns all of it to the driver.  Safe to call at any time no render is in flight.
 * RM_TRACE=1 in the environment prints the phase timings of rm_render_tiled / the render driver on stderr. */
int rm_release_cached_memory(void);

/* Tile rectangles in the reference's queue order (column-major: y advances
 * first, edge tiles clipped — src/trace.rs:142-173).  Returns the tile count;
 * writes min(count, capacity) entries of {left, top, width, height}. */
size_t rm_tile_layout(const rm_settings* settings, size_t* rects, size_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* RAYMOND_H */
