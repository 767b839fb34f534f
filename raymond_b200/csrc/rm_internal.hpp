// rm_internal.hpp — host-side object model behind include/raymond.h (not part of the ABI).
#pragma once

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <condition_variable>
#include <cstdint>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/raymond.h"

struct rm_renderer;

namespace rm {

void set_error(const std::string& msg);
int fail(int status, const std::string& msg);
// RM_ERR_INVALID_ARGUMENT for camera settings the reference's camera could not finish or would panic on (D2, D6); no device work
int validate_camera(const rm_camera_settings& c, const char* who);

// Mesh { triangles, bounding_box }                         reference core/src/geometry/mesh.rs:10-13
struct Mesh {
    std::vector<rm_triangle> triangles;
    rm_aabb bounds;
};
rm_aabb mesh_bounds(const rm_triangle* tris, size_t n);    // Mesh::find_mesh_bounds  mesh.rs:123-140

// AccGrid in compressed-row form.  The reference keeps `cells` (offset into
// `mapping_table`) and `mapping_table` ([count, tri...] per cell, acc_grid.rs:67-74);
// here the same per-cell lists, in the same ascending-triangle order, are stored
// as cell_start[c]..cell_start[c+1] into `references`.
// Page-locked host staging blocks, cached across calls (pinning is the expensive part of a short upload).
// Defined in rm_device.cu.  acquire() returns nullptr when pinning fails.
void* pinned_acquire(size_t bytes);
void pinned_release(void* p);

struct Grid {
    std::vector<rm_triangle> triangles;
    rm_aabb bounds;
    uint64_t resolution[3];
    rm_vec3 cell_size;
    std::vector<uint32_t> cell_start;   // n_cells + 1
    std::vector<uint32_t> references;   // triangle indices
    uint64_t n_cells() const { return resolution[0] * resolution[1] * resolution[2]; }
    // The grid as the device wants it (prepare_grid_image's host image), kept in pinned memory after the first upload so that
    // every later upload of this immutable grid is one H2D copy with no flattening.  Only for images <= kImageCacheLimit.
    mutable std::mutex image_mu;
    mutable void* image = nullptr;
    mutable size_t image_bytes = 0;
    Grid() = default;
    Grid(const Grid&) = delete;
    Grid& operator=(const Grid&) = delete;
    ~Grid() { if (image) { pinned_release(image); g_grid_image_bytes -= image_bytes; } }
    static std::atomic<size_t> g_grid_image_bytes;      // pinned bytes held by all grids' images (rm_device.cu)
};
constexpr size_t kImageCacheLimit = (size_t)2 << 30;          // largest image kept with its grid
constexpr size_t kImageCacheTotalLimit = (size_t)8 << 30;     // ... and how much all grids together may keep pinned
// AccGrid::build_from_mesh                                 acc_grid.rs:36-83
int grid_dims(const rm_aabb& bounds, size_t n, uint64_t res[3], double cell[3]);
int build_grid(std::vector<rm_triangle>&& tris, const rm_aabb& bounds, std::shared_ptr<Grid>* out);
// the same, with the cell lists counted, scanned and filled on the GPU (rm_gridbuild.cu)
int build_grid_device(std::vector<rm_triangle>&& tris, const rm_aabb& bounds, int device, std::shared_ptr<Grid>* out);

enum GeometryKind : int { GEOM_PLANE = 0, GEOM_SPHERE = 1, GEOM_GRID = 2 };   // scene.rs:9-13

// The colour texture of one object (rm_scene_set_texture), immutable once set: width x height texels, row 0 = top, stored as
// RGBA f32 (A = 0) in the layout the device reads.  Scenes and the placements made from them share it.
struct Texture {
    std::vector<float> rgba;
    size_t width = 0, height = 0;
    double scale_u = 1.0, scale_v = 1.0;
};

struct Object {                                             // scene.rs:33-37
    int geometry;
    rm_vec3 origin;
    rm_vec3 normal;
    double radius;
    std::shared_ptr<Grid> grid;
    rm_material material;
    std::shared_ptr<const Texture> texture;                 // none in the reference: null = the material's one colour
};

// The environment map of a scene (rm_scene_set_environment), immutable once set: width x height texels, row 0 = +y, stored as
// RGBA f32 (A = 0) in the layout the device reads.  Scenes and the placements made from them share it.
struct Environment {
    std::vector<float> rgba;
    size_t width = 0, height = 0;
    double scale = 1.0, rotation = 0.0;
};

struct TileRect { size_t left, top, width, height; };
// tile split of render_tiled                               src/trace.rs:142-173
std::vector<TileRect> tile_layout(size_t W, size_t H, size_t tw, size_t th);

// The part of a frame one share renders (rm_gpu_options rank / world_size / partition): share `rank` of `world` owns the tiles
// t with t % world == rank under RM_PARTITION_TILES, and the global samples rank, rank + world, ... of every pixel under
// RM_PARTITION_SAMPLES.  world_size <= 1, or any other partition value, is the whole frame.
struct Share {
    size_t rank = 0, world = 1;
    bool tiles = false;
    explicit Share(const rm_gpu_options& o) {
        if (o.world_size > 1 && (o.partition == RM_PARTITION_SAMPLES || o.partition == RM_PARTITION_TILES)) {
            rank = (size_t)o.rank;
            world = (size_t)o.world_size;
            tiles = o.partition == RM_PARTITION_TILES;
        }
    }
    // owned tiles: first_tile(), first_tile() + tile_step(), ... of the layout
    size_t first_tile() const { return tiles ? rank : 0; }
    size_t tile_step() const { return tiles ? world : 1; }
    bool owns_tile(size_t t) const { return t % tile_step() == first_tile(); }
    // the global samples of [begin, end) this share renders: *count of them from *first, sample_stride() apart
    size_t sample_stride() const { return tiles ? 1 : world; }
    void samples(size_t begin, size_t end, size_t* first, size_t* count) const {
        const size_t G = sample_stride();
        *first = begin + (rank + G - begin % G) % G;
        *count = *first < end ? (end - *first + G - 1) / G : 0;
    }
};

// Sum of the accumulators of several renderers (one per share of a task) into a host frame (rm_device.cu).  With a pinned
// destination every device sums its slice of the frame from all peers' accumulators in place (peer reads over NVLink) and
// writes it straight to the host; otherwise the sums are gathered onto the first device and copied.  Either way the sum
// is taken in renderer order, the renderers' accumulators are left as they are, and on return the frame is complete.
// `mean_pinned` (optional, pinned): the peer-memory path also writes sum / divisor there (the finalize of await(), fused into
// the exchange) and sets *mean_written; the other paths leave it alone.
int reduce_accumulators_to_host(rm_renderer* const* renderers, int count, rm_vec3* out, bool out_is_pinned, rm_vec3* mean_pinned = nullptr,
                                double divisor = 1.0, bool* mean_written = nullptr);
// E_t (include/raymond.h) of tiles first, first + step, ... after `n` samples from the S and Q summed over the renderers
// (RM_FLAG_MOMENTS) in renderer order, into `out_pinned` (a pinned_acquire block of n_tiles doubles; other tiles are left
// alone).  Device g computes every count-th of those tiles from the g-th on, reading its peers' sums in place; without peer
// mappings the sums are staged onto the first device.  Synchronous.
int tile_errors_to_host(rm_renderer* const* renderers, int count, size_t n, double* out_pinned, size_t n_tiles, size_t first, size_t step);
// display transform kernel (rm_display.cu): sums / divisor -> tonemap -> 8-bit RGB, device pointers
int tonemap_device(const double* sums_device, size_t n_pixels, double divisor, double exposure, double gamma, unsigned char* out_device, void* stream);

// ---- the a-trous denoiser of rm_renderer_read_denoised and rm_render_tiled_denoised (kernels in rm_display.cu)
// `settings` NULL = the defaults of include/raymond.h; RM_ERR_INVALID_ARGUMENT (no device work) for iterations outside 1..10 or a
// sigma the f32 filter cannot use.  `who` names the entry point in the message.
int resolve_denoise_settings(const rm_denoise_settings* settings, rm_denoise_settings* out, const char* who);
// The whole filter on one device: from the device sums S, Q and the RM_FLAG_AOV planes of a W x H frame after n samples to W*H
// denoised means, written as f64 by the last pass into `out_mapped` (the device address of a pinned, mapped host frame), on `stream`.
// Synchronous; launches 1 + s.iterations kernels.
int denoise_to_host(const double* sums, const double* moments, const double* aov, size_t W, size_t H, double n, const rm_denoise_settings& s,
                    rm_vec3* out_mapped, void* stream);
// The same filter with the frame sliced by rows over the shares of a task: share g of count owns rows [H*g/count, H*(g+1)/count).
// Every share's sums (whole-frame planes, zeros where it rendered nothing) and packed rows are read in place by the other shares'
// kernels (peer mappings): `packed[g]` holds 4 planes of (rows of g) * W float4 — colour + variance ping, pong, albedo + depth,
// normal — from the peer-visible block cache.
constexpr int kMaxShares = 64;      // pointers one kernel parameter block takes per kind of buffer
struct DenoiseSlices {
    const double* sums[kMaxShares];
    const double* moments[kMaxShares];
    const double* aov[kMaxShares];
    void* packed[kMaxShares];
    int count;
};
#ifdef __CUDACC__
__host__ __device__
#endif
inline size_t slice_begin(size_t H, size_t g, size_t count) { return H * g / count; }
// Launchers of one share's part (0 = launched or nothing to do, else a cudaError_t value).  denoise_reduce_slice: its rows of S, Q and
// the features summed over all shares in share order, packed as the one-device filter packs them.  denoise_pass_slice: pass `pass`
// (step 2^pass) of its rows, taps read from whichever share owns them; `out_mapped` non-NULL: the result goes there as f64 instead.
int denoise_reduce_slice(const DenoiseSlices& d, int share, size_t W, size_t H, double n, void* stream);
int denoise_pass_slice(const DenoiseSlices& d, int share, size_t W, size_t H, uint32_t pass, const rm_denoise_settings& s, rm_vec3* out_mapped,
                       void* stream);
// The filter over the sums of several renderers (rm_device.cu; one renderer: rm_renderer_read_denoised).  Sliced as above when every
// device maps every other's memory and count <= kMaxShares; otherwise S, Q and the features are staged onto the first device and the
// one-device filter runs there.  The W*H result lands in `out_pinned` (a pinned_acquire block).  Synchronous.
int denoise_shares_to_host(rm_renderer* const* renderers, int count, size_t n, const rm_denoise_settings& s, rm_vec3* out_pinned);
// Device memory from the cached stream-ordered pool (rm_device.cu); dev_alloc returns a cudaError_t value (0 = ok).
int dev_alloc(void** p, size_t bytes);
void dev_release(void* p);

// RM_TRACE=1 in the environment: phase timings of rm_render_tiled / the render driver on stderr (host-path tuning)
struct Trace {
    bool on;
    std::chrono::steady_clock::time_point t0;
    Trace() : on(getenv("RM_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what) const {
        if (on) fprintf(stderr, "[rm_trace] %8.3f ms  %s\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(), what);
    }
};

}  // namespace rm

// internal entry points of rm_device.cu used by the task driver (C linkage, not part of include/raymond.h)
extern "C" {
rm_renderer* rm_renderer_create_unbound(const rm_settings* settings, const rm_gpu_options* options);
// a scene placed on one device or several at once (slices over every device's PCIe link + an all-gather over NVLink): one host thread
// per share calls _join, ALL shares must; _join returns the share's device scene or NULL
struct rm_scene_group;
rm_scene_group* rm_scene_group_create(const rm_scene* scene, const int32_t* devices, int count);
rm_device_scene* rm_scene_group_join(rm_scene_group* group, int share);
void rm_scene_group_destroy(rm_scene_group* group);
int rm_renderer_bind_scene(rm_renderer* r, rm_device_scene* ds, int owning);
rm_device_scene* rm_renderer_device_scene(rm_renderer* r);
// the coverage mask of the camera rays (DESIGN §3.7), W*H ints 0 / 1; RM_ERR_STATE when the renderer has none
int rm_renderer_coverage(rm_renderer* r, int32_t* out_host);
}

struct rm_mesh { rm::Mesh mesh; };
struct rm_grid { std::shared_ptr<rm::Grid> grid; std::atomic<int> refs{1}; };
struct rm_scene { std::vector<rm::Object> objects; std::shared_ptr<const rm::Environment> env; };
