// rm_device.cu — host plumbing of the GPU path: scene flattening + upload, launch sequencing of the
// wavefront stages (kernels in rm_kernels.cuh), the accumulator, and the device-level C ABI.
// Citations are relative to the reference checkout (Nyrox/raymond).

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <type_traits>
#include <vector>

#include "rm_kernels.cuh"

namespace rm {

#define RM_CUDA(call)                                                                                   \
    do {                                                                                                \
        cudaError_t e__ = (call);                                                                       \
        if (e__ != cudaSuccess)                                                                         \
            return fail(RM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));              \
    } while (0)

static int sm_count(int device) {
    int n = 148;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device);
    return n > 0 ? n : 148;
}

// RM_OK, or RM_ERR_CUDA when `device` is not the ordinal of a CUDA device of this process
static int check_device(int device) {
    int count = 0;
    const cudaError_t e = cudaGetDeviceCount(&count);
    if (e == cudaSuccess && device >= 0 && device < count) return RM_OK;
    return fail(RM_ERR_CUDA, std::string("no usable CUDA device ") + std::to_string(device) + " (" + (e != cudaSuccess ? cudaGetErrorString(e) : "ordinal out of range") +
                                 "); this library has no CPU path");
}

// ---- device memory: stream-ordered allocations from a PRIVATE pool per device (the device's default pool, which torch and
// other libraries in the process may use, is left alone).  The pool keeps up to kPoolKeepBytes of freed memory mapped, so the
// multi-GB wavefront queues of one render are handed to the next one instead of being unmapped and re-mapped (cudaFree /
// cudaMalloc of 10 GB cost 0.1-0.5 s each); anything beyond that goes back to the driver at the next synchronisation, and
// rm_release_cached_memory() returns all of it.  The pool is private to its device (granting peers access to a whole pool made
// growing it fail on multi-GPU boxes); the one buffer peers read directly — the accumulator — is a plain cudaMalloc
// allocation, reachable through cudaDeviceEnablePeerAccess.  All pool traffic is ordered on the legacy default stream; users
// synchronise their own stream before dev_free().
namespace {
constexpr unsigned long long kPoolKeepBytes = 48ull << 30;
std::mutex g_pool_mu;
std::map<int, cudaMemPool_t> g_pools;
}  // namespace

static cudaError_t device_pool(int dev, cudaMemPool_t* out) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    auto it = g_pools.find(dev);
    if (it != g_pools.end()) { *out = it->second; return cudaSuccess; }
    cudaMemPoolProps props{};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool = nullptr;
    cudaError_t e = cudaMemPoolCreate(&pool, &props);
    if (e != cudaSuccess) return e;
    unsigned long long keep = kPoolKeepBytes;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    cudaGetLastError();
    g_pools[dev] = pool;
    *out = pool;
    return cudaSuccess;
}

static cudaError_t dev_malloc_raw(void** p, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    cudaMemPool_t pool = nullptr;
    if (e == cudaSuccess) e = device_pool(dev, &pool);
    if (e == cudaSuccess) e = cudaMallocFromPoolAsync(p, std::max<size_t>(bytes, 32), pool, 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    if (e == cudaErrorMemoryAllocation && pool) {
        // say what the device and the pool hold: an out-of-memory here is usually memory cached or in use elsewhere in the process
        size_t free_b = 0, total_b = 0;
        unsigned long long reserved = 0, used = 0;
        cudaGetLastError();
        cudaMemGetInfo(&free_b, &total_b);
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved);
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
        fprintf(stderr, "[raymond] device %d: allocation of %zu bytes failed; device free %zu of %zu, pool reserved %llu, pool in use %llu\n", dev, bytes, free_b,
                total_b, reserved, used);
        cudaGetLastError();
    }
    return e;
}
template <typename T>
static cudaError_t dev_malloc(T** p, size_t bytes) { return dev_malloc_raw((void**)p, bytes); }
static void dev_free(void* p) { if (p) cudaFreeAsync(p, 0); }

int dev_alloc(void** p, size_t bytes) { return (int)dev_malloc_raw(p, bytes); }
void dev_release(void* p) { dev_free(p); }

// ---- peer-visible blocks: what other devices of the process read in place — the accumulators (the exchange kernel of a
// multi-device task) and the scene blocks (the all-gather of a scene placed on several devices) — are plain cudaMalloc
// allocations, reachable through cudaDeviceEnablePeerAccess, and are kept per (device, size) for the next frame: with peer
// access on, cudaMalloc / cudaFree map and unmap on every peer and cost milliseconds.
namespace {
struct VisibleBlock { int device; size_t bytes; void* p; };
std::mutex g_visible_mu;
std::vector<VisibleBlock>& g_visible_free = *new std::vector<VisibleBlock>();      // never destroyed (it frees device memory)
constexpr size_t kVisibleCacheBytes = (size_t)16 << 30;
}  // namespace

static cudaError_t visible_acquire(int device, size_t bytes, void** out) {
    {
        std::lock_guard<std::mutex> lk(g_visible_mu);
        for (size_t i = 0; i < g_visible_free.size(); i++)
            if (g_visible_free[i].device == device && g_visible_free[i].bytes == bytes) {
                *out = g_visible_free[i].p;
                g_visible_free.erase(g_visible_free.begin() + (long)i);
                return cudaSuccess;
            }
    }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e == cudaErrorMemoryAllocation) {          // make room: drop what is cached, then once more
        cudaGetLastError();
        std::vector<VisibleBlock> drop;
        { std::lock_guard<std::mutex> lk(g_visible_mu); drop.swap(g_visible_free); }
        for (const VisibleBlock& b : drop) { cudaSetDevice(b.device); cudaFree(b.p); }
        cudaSetDevice(device);
        e = cudaMalloc(out, bytes);
    }
    return e;
}

static void visible_release(int device, size_t bytes, void* p) {      // the caller's work on `p` is complete
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(g_visible_mu);
        size_t cached = 0;
        for (const VisibleBlock& b : g_visible_free) cached += b.bytes;
        if (cached + bytes <= kVisibleCacheBytes) { g_visible_free.push_back({device, bytes, p}); return; }
    }
    cudaSetDevice(device);
    cudaFree(p);
}

static void visible_cache_clear() {
    std::vector<VisibleBlock> drop;
    { std::lock_guard<std::mutex> lk(g_visible_mu); drop.swap(g_visible_free); }
    for (const VisibleBlock& b : drop) { cudaSetDevice(b.device); cudaFree(b.p); }
}

// device `from` may read the memory of device `to` in place (a no-op after the first time; false when the hardware cannot)
static bool enable_peer(int from, int to) {
    if (from == to) return true;
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, from, to) != cudaSuccess || !can) { cudaGetLastError(); return false; }
    if (cudaSetDevice(from) != cudaSuccess) { cudaGetLastError(); return false; }
    const cudaError_t e = cudaDeviceEnablePeerAccess(to, 0);
    cudaGetLastError();
    return e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled;
}

// ---- pinned staging pool
namespace {
struct PinnedBlock { void* p; size_t bytes; };
std::mutex g_pin_mu;
std::vector<PinnedBlock> g_pin_free, g_pin_busy;
constexpr size_t kPinnedCacheLimit = (size_t)8 << 30;      // blocks beyond 8 GiB of cache are unpinned on release
}  // namespace

std::atomic<size_t> Grid::g_grid_image_bytes{0};

void* pinned_acquire(size_t bytes) {
    bytes = std::max<size_t>(bytes, 4096);
    std::lock_guard<std::mutex> lk(g_pin_mu);
    size_t best = g_pin_free.size();
    for (size_t i = 0; i < g_pin_free.size(); i++)
        if (g_pin_free[i].bytes >= bytes && (best == g_pin_free.size() || g_pin_free[i].bytes < g_pin_free[best].bytes)) best = i;
    PinnedBlock b{nullptr, 0};
    if (best != g_pin_free.size()) {
        b = g_pin_free[best];
        g_pin_free.erase(g_pin_free.begin() + (long)best);
    } else {
        // drop cached blocks that are too small before pinning a bigger one
        for (PinnedBlock& f : g_pin_free) cudaFreeHost(f.p);
        g_pin_free.clear();
        // portable + mapped: every device of the process can DMA from it and write to it from a kernel (the accumulator exchange does)
        if (cudaHostAlloc(&b.p, bytes, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        b.bytes = bytes;
    }
    g_pin_busy.push_back(b);
    return b.p;
}

void pinned_release(void* p) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_pin_mu);
    for (size_t i = 0; i < g_pin_busy.size(); i++)
        if (g_pin_busy[i].p == p) {
            PinnedBlock b = g_pin_busy[i];
            g_pin_busy.erase(g_pin_busy.begin() + (long)i);
            size_t cached = 0;
            for (const PinnedBlock& f : g_pin_free) cached += f.bytes;
            if (cached + b.bytes <= kPinnedCacheLimit) g_pin_free.push_back(b);
            else cudaFreeHost(b.p);
            return;
        }
}

static DevCamera make_camera(const rm_camera_settings& c) {
    DevCamera d{};
    d.pos[0] = c.position.x; d.pos[1] = c.position.y; d.pos[2] = c.position.z;
    d.width = (double)c.backbuffer_width;
    d.height = (double)c.backbuffer_height;
    d.aspect = d.width / d.height;
    d.tan_half = std::tan(c.fov_vert / 2.0 * 3.14159265358979323846 / 180.0);   // src/trace.rs:329-330
    d.focal_length = c.focal_length;
    d.aperture_radius = c.aperture_radius;
    d.W = (int)c.backbuffer_width;
    d.H = (int)c.backbuffer_height;
    d.use_dof = c.aperture_radius > 0.0 ? 1 : 0;   // the reference's DoF loop never ends for radius 0
    return d;
}

// Owned pixels of a share in launch order, resident on one device (see pixel_map_for).
struct PixelMap {
    unsigned* dev = nullptr;
    size_t n = 0;
    int device = 0;
    ~PixelMap();
};

// Device buffers one batch of rays needs for Scene::intersect: hit records and the traversal queue.
struct IntersectBuffers {
    HitArrays hit{};
    double* trav = nullptr;
    size_t cap = 0;
    int alloc(size_t n) {
        cap = std::max<size_t>(n, 32);
        RM_CUDA(dev_malloc(&hit.t, cap * sizeof(double)));
        RM_CUDA(dev_malloc(&hit.obj, cap * sizeof(int)));
        RM_CUDA(dev_malloc(&hit.sub, cap * sizeof(unsigned)));
        RM_CUDA(dev_malloc(&trav, cap * kTravDoubles * sizeof(double)));
        return RM_OK;
    }
    void release() {
        dev_free(hit.t); dev_free(hit.obj); dev_free(hit.sub); dev_free(trav);
        hit = HitArrays{}; trav = nullptr; cap = 0;
    }
};

}  // namespace rm

using namespace rm;

// --------------------------------------------------------------------- device scene

struct rm_device_scene {
    int device = 0;
    int sms = 148;
    int traverse_blocks_per_sm = 2;
    DevScene scene{};
    std::vector<int> grid_objects;          // object indices with Geometry::Grid, ascending
    const float4* tri_spheres[kMaxGrids] = {};  // per distinct grid: one bounding sphere per triangle (§3.1), in the grid's block ...
    size_t n_triangles[kMaxGrids] = {};     // ... and its triangle count
    bool emissive_grid = false;             // a grid object has an Emission material: its traversal can decide a last-depth path
    bool has_env = false;                   // the scene has an environment map: `env` points at this device's copy of its texels
    DevEnv env{};
    bool has_tex = false;                   // an object has a colour texture: `tex` points at this device's copies
    DevTex tex{};
    std::vector<void*> allocations;         // one device block per distinct grid, in DevScene::grid order, then the environment map,
                                            // the textures in object order and the uvs of the textured grids
    std::vector<size_t> allocation_bytes;
    std::vector<std::shared_ptr<Grid>> keep;
    double upload_ms = 0.0;
    size_t bytes = 0;
    // scratch of rm_device_scene_intersect (grow-only)
    std::mutex query_mu;
    IntersectBuffers query;
    unsigned* query_counters = nullptr;     // {traversal records, traversal cursor}
    cudaEvent_t query_done = nullptr;       // end of the last query: the next one (on whatever stream) waits for it before it reuses the scratch
    ~rm_device_scene() {
        cudaSetDevice(device);
        cudaDeviceSynchronize();            // queries may still be running on the caller's streams
        if (query_done) cudaEventDestroy(query_done);
        for (size_t i = 0; i < allocations.size(); i++) visible_release(device, allocation_bytes[i], allocations[i]);
        query.release();
        dev_free(query_counters);
    }
};

namespace rm {

__global__ void __launch_bounds__(256) k_spread_spheres(const float4* __restrict__ per_triangle, const unsigned* __restrict__ refs, size_t n_refs,
                                                         float4* __restrict__ per_reference) {
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_refs; p += (size_t)gridDim.x * blockDim.x)
        per_reference[p] = __ldg(&per_triangle[__ldg(&refs[p])]);
}

// One sphere per occupied cell (DevGrid::csph) from the per-reference spheres of its list: f32 centre at the middle of the box
// around the members' spheres, radius R_c >= (max |c_c - c_i| + R_i) (1 + 2e-6), evaluated in f64 and rounded up to f32, so that
// every member sphere lies inside it with the margin DESIGN §3.1 needs; a member with a non-finite radius (a non-finite triangle)
// makes the cell's infinite (never culled).  Empty cells are never read and get an infinite one.
__global__ void __launch_bounds__(256) k_cell_spheres(const uint2* __restrict__ cells, size_t n_cells, const float4* __restrict__ sphr,
                                                       float4* __restrict__ csph) {
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_cells; c += (size_t)gridDim.x * blockDim.x) {
        const uint2 cell = __ldg(&cells[c]);
        double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        bool finite = cell.y > 0;
        for (unsigned p = cell.x; p < cell.x + cell.y; p++) {
            const float4 m = __ldg(&sphr[p]);
            const double r = (double)m.w;
            finite = finite && isfinite(r);
            lo[0] = fmin(lo[0], (double)m.x - r); hi[0] = fmax(hi[0], (double)m.x + r);
            lo[1] = fmin(lo[1], (double)m.y - r); hi[1] = fmax(hi[1], (double)m.y + r);
            lo[2] = fmin(lo[2], (double)m.z - r); hi[2] = fmax(hi[2], (double)m.z + r);
        }
        const float cx = (float)((lo[0] + hi[0]) * 0.5), cy = (float)((lo[1] + hi[1]) * 0.5), cz = (float)((lo[2] + hi[2]) * 0.5);
        double reach = 0.0;
        for (unsigned p = cell.x; finite && p < cell.x + cell.y; p++) {
            const float4 m = __ldg(&sphr[p]);
            const double dx = (double)cx - (double)m.x, dy = (double)cy - (double)m.y, dz = (double)cz - (double)m.z;
            reach = fmax(reach, sqrt((dx * dx + dy * dy) + dz * dz) + (double)m.w);
        }
        const float rc = __double2float_ru(reach * (1.0 + 2e-6));
        csph[c] = finite && isfinite(rc) && isfinite(cx) && isfinite(cy) && isfinite(cz) ? make_float4(cx, cy, cz, rc)
                                                                                          : make_float4(0.f, 0.f, 0.f, INFINITY);
    }
}

// The flattened image of one grid: the arrays of DevGrid laid out in ONE block — [tri][shd][cells][occ][refs][one sphere per
// triangle] come from the host, [one sphere per reference] behind them is spread on the device (k_spread_spheres), so it never
// crosses the bus.  The host image of an immutable grid is built once by a few host threads and kept (pinned) with the grid;
// images above kImageCacheLimit are staged through a pooled pinned block per upload.
struct GridImage {
    DevGrid header{};          // geometry of the grid; the array pointers are set by point_grid()
    size_t off_tri = 0, off_shd = 0, off_cells = 0, off_occ = 0, off_refs = 0, off_spht = 0, host_total = 0, off_sph = 0, total = 0, nr = 0, nt = 0;
    size_t off_csph = 0, nc = 0;    // one sphere per cell behind them (none with RM_NO_CELL_SPHERES when the image was laid out)
    char* host = nullptr;
    bool cached = false;       // the host image belongs to the grid (not released after the upload)
};

static int prepare_grid_image(const Grid& g, GridImage* out) {
    GridImage& im = *out;
    DevGrid& d = im.header;
    d.bmin[0] = g.bounds.min.x; d.bmin[1] = g.bounds.min.y; d.bmin[2] = g.bounds.min.z;
    d.bmax[0] = g.bounds.max.x; d.bmax[1] = g.bounds.max.y; d.bmax[2] = g.bounds.max.z;
    d.cell[0] = g.cell_size.x; d.cell[1] = g.cell_size.y; d.cell[2] = g.cell_size.z;
    for (int a = 0; a < 3; a++) d.res[a] = (int)g.resolution[a];
    const double ex = d.bmax[0] - d.bmin[0], ey = d.bmax[1] - d.bmin[1], ez = d.bmax[2] - d.bmin[2];
    d.diag2 = ex * ex + ey * ey + ez * ez;
    d.diag = std::sqrt(d.diag2);
    d.n_cells = g.n_cells();
    const size_t nc = (size_t)d.n_cells, nt = g.triangles.size(), nr = g.references.size();
    const size_t n_occ = (nc + 31) / 32;
    auto pad = [](size_t b) { return (b + 255) & ~(size_t)255; };
    im.nr = nr;
    im.nt = nt;
    im.off_tri = 0;
    im.off_shd = im.off_tri + pad(nt * 12 * sizeof(double));
    im.off_cells = im.off_shd + pad(nt * 18 * sizeof(double));
    im.off_occ = im.off_cells + pad(nc * sizeof(uint2));
    im.off_refs = im.off_occ + pad(n_occ * sizeof(unsigned));
    im.off_spht = im.off_refs + pad(nr * sizeof(unsigned));
    im.host_total = im.off_spht + pad(nt * sizeof(float4)) + 256;
    im.off_sph = im.host_total;
    im.total = im.off_sph + pad(nr * sizeof(float4)) + 256;
    im.nc = nc;
    if (getenv("RM_NO_CELL_SPHERES") == nullptr) {
        im.off_csph = im.total;
        im.total = im.off_csph + pad(nc * sizeof(float4)) + 256;
    }
    const size_t host_total = im.host_total;
    std::unique_lock<std::mutex> image_lock(g.image_mu);
    const bool have_image = g.image && g.image_bytes == host_total;
    const bool keep_image = have_image || (host_total <= kImageCacheLimit && Grid::g_grid_image_bytes.load() + host_total <= kImageCacheTotalLimit);
    if (!keep_image) image_lock.unlock();
    char* host = have_image ? (char*)g.image : (char*)pinned_acquire(host_total);
    if (!host) return fail(RM_ERR_OUT_OF_MEMORY, "cannot pin " + std::to_string(host_total) + " bytes of host staging memory");
    im.host = host;
    im.cached = keep_image;
    if (have_image) return RM_OK;
    double* tri = (double*)(host + im.off_tri);
    double* shd = (double*)(host + im.off_shd);
    float4* sph_tri = (float4*)(host + im.off_spht);      // one bounding sphere per triangle
    uint2* cells = (uint2*)(host + im.off_cells);
    unsigned* occ = (unsigned*)(host + im.off_occ);
    unsigned* refs = (unsigned*)(host + im.off_refs);

    auto fill_triangles = [&](size_t lo, size_t hi) {
        for (size_t i = lo; i < hi; i++) {
            const rm_triangle& t = g.triangles[i];
            const rm_vertex* v[3] = {&t.v0, &t.v1, &t.v2};
            double* tp = tri + i * 12;
            double* sp = shd + i * 18;
            for (int k = 0; k < 3; k++) {
                tp[3 * k + 0] = v[k]->position.x; tp[3 * k + 1] = v[k]->position.y; tp[3 * k + 2] = v[k]->position.z;
                sp[3 * k + 0] = v[k]->position.x; sp[3 * k + 1] = v[k]->position.y; sp[3 * k + 2] = v[k]->position.z;
                sp[9 + 3 * k + 0] = v[k]->normal.x; sp[9 + 3 * k + 1] = v[k]->normal.y; sp[9 + 3 * k + 2] = v[k]->normal.z;
            }
            tp[9] = tp[10] = tp[11] = 0.0;
            // bounding sphere for the conservative pre-test (cull_sphere): f32 centre near the centre of the vertices' box,
            // radius to the farthest vertex measured from that f32 centre, inflated and rounded up; a non-finite triangle
            // gets an infinite radius (never culled)
            float cf[3];
            double cmax = 0.0, r2 = 0.0;
            for (int a = 0; a < 3; a++) {
                const double lo = std::fmin(tp[a], std::fmin(tp[3 + a], tp[6 + a])), hi = std::fmax(tp[a], std::fmax(tp[3 + a], tp[6 + a]));
                cf[a] = (float)(0.5 * (lo + hi));
                cmax = std::fmax(cmax, std::fabs((double)cf[a]));
            }
            for (int k = 0; k < 3; k++) {
                const double dx = tp[3 * k] - (double)cf[0], dy = tp[3 * k + 1] - (double)cf[1], dz = tp[3 * k + 2] - (double)cf[2];
                r2 = std::fmax(r2, dx * dx + dy * dy + dz * dz);
            }
            const double r = std::sqrt(r2) * (1.0 + 1e-6) + 1e-9 * (1.0 + cmax);
            float rf = (float)r;
            if (!((double)rf >= r)) rf = std::nextafterf(rf, INFINITY);
            if (!(r == r) || !std::isfinite(cf[0]) || !std::isfinite(cf[1]) || !std::isfinite(cf[2])) { cf[0] = cf[1] = cf[2] = 0.f; rf = INFINITY; }
            sph_tri[i] = make_float4(cf[0], cf[1], cf[2], rf);
        }
    };
    auto fill_cells = [&](size_t lo, size_t hi) {      // lo, hi multiples of 32 (whole occupancy words)
        for (size_t w = lo / 32; w < (hi + 31) / 32; w++) {
            unsigned bits = 0;
            for (size_t c = w * 32; c < std::min(w * 32 + 32, nc); c++) {
                const unsigned count = g.cell_start[c + 1] - g.cell_start[c];
                cells[c] = make_uint2(g.cell_start[c], count);
                if (count) bits |= 1u << (c & 31);
            }
            occ[w] = bits;
        }
    };
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t workers = (nt + nc + nr < ((size_t)1 << 18)) ? 1 : std::min<size_t>(hw ? hw : 4, 8);
    std::vector<std::thread> pool;
    for (size_t w = 1; w < workers; w++)
        pool.emplace_back([&, w] {
            fill_triangles(nt * w / workers, nt * (w + 1) / workers);
            fill_cells((nc * w / workers) & ~(size_t)31, w + 1 == workers ? nc : (nc * (w + 1) / workers) & ~(size_t)31);
        });
    fill_triangles(0, nt / workers);
    fill_cells(0, workers == 1 ? nc : (nc / workers) & ~(size_t)31);
    if (nr) memcpy(refs, g.references.data(), nr * sizeof(unsigned));
    for (std::thread& t : pool) t.join();
    if (keep_image) { g.image = host; g.image_bytes = host_total; Grid::g_grid_image_bytes += host_total; }
    return RM_OK;
}

static void release_grid_image(GridImage& im) {
    if (im.host && !im.cached) pinned_release(im.host);
    im.host = nullptr;
}

static void point_grid(const GridImage& im, void* dev, DevGrid* out) {
    DevGrid d = im.header;
    d.tri = (const double*)((char*)dev + im.off_tri);
    d.shd = (const double*)((char*)dev + im.off_shd);
    d.sphr = (const float4*)((char*)dev + im.off_sph);
    d.cells = (const uint2*)((char*)dev + im.off_cells);
    d.occ = (const unsigned*)((char*)dev + im.off_occ);
    d.refs = (const unsigned*)((char*)dev + im.off_refs);
    d.csph = im.off_csph ? (const float4*)((char*)dev + im.off_csph) : nullptr;
    *out = d;
}

// one sphere per REFERENCE, in reference order: a cell's candidates become one contiguous read for k_traverse
static cudaError_t spread_spheres(const GridImage& im, void* dev, int sms, cudaStream_t stream) {
    if (!im.nr) return cudaSuccess;
    k_spread_spheres<<<(unsigned)std::min<size_t>((im.nr + 255) / 256, (size_t)sms * 32), 256, 0, stream>>>(
        (const float4*)((char*)dev + im.off_spht), (const unsigned*)((char*)dev + im.off_refs), im.nr, (float4*)((char*)dev + im.off_sph));
    if (!im.off_csph || !im.nc) return cudaGetLastError();
    k_cell_spheres<<<(unsigned)std::min<size_t>((im.nc + 255) / 256, (size_t)sms * 32), 256, 0, stream>>>(
        (const uint2*)((char*)dev + im.off_cells), im.nc, (const float4*)((char*)dev + im.off_sph), (float4*)((char*)dev + im.off_csph));
    return cudaGetLastError();
}

}  // namespace rm

// --------------------------------------------------------------------- placing a scene on its devices
//
// A scene goes onto one device or onto the devices of several shares at once: the host image of every grid crosses the bus
// ONCE, in slices — share g copies slice g to its own device over its own PCIe link — and every share then pulls the other
// slices from its peers over NVLink (an all-gather of the image); the per-reference spheres are spread on every device
// locally.  One host thread per share calls rm_scene_group_join; all of them must.
struct rm_scene_group {
    std::vector<int> devices;
    DevScene table{};                               // every share's object table; the grid arrays are pointed per share
    std::vector<int> grid_objects;                  // object indices with Geometry::Grid, ascending
    bool emissive_grid = false;
    std::shared_ptr<const Environment> env;         // the scene's environment map (or none); every share uploads its own copy
    std::vector<std::shared_ptr<const Texture>> textures;   // per object: its colour texture (or none); every share uploads its own copies
    std::vector<std::vector<double>> grid_uv;       // per distinct grid: 6 f64 per triangle (uv0 uv1 uv2) when a textured object references it
    std::vector<std::shared_ptr<Grid>> grids;       // distinct grids, in DevScene::grid order
    std::vector<GridImage> images;                  // ... and their host images
    double flatten_ms = 0.0;                        // host time of the table and the images
    std::mutex mu;
    std::condition_variable cv;
    std::vector<std::vector<void*>> blocks;         // [share][grid]: the share's device block
    std::vector<cudaEvent_t> uploaded;              // [share]: its slice of every grid is on its device
    int arrived[2] = {0, 0};                        // shares that reached barrier 0 (slices uploaded) / 1 (gather done)
    bool failed = false;

    // every share arrives exactly once per barrier, also after a failure of its own (so nobody waits forever)
    bool barrier(int which, bool ok) {
        std::unique_lock<std::mutex> lk(mu);
        if (!ok) failed = true;
        arrived[which]++;
        cv.notify_all();
        cv.wait(lk, [&] { return arrived[which] >= (int)devices.size(); });
        return !failed;
    }
    ~rm_scene_group() {
        for (GridImage& im : images) release_grid_image(im);
        for (cudaEvent_t e : uploaded) if (e) cudaEventDestroy(e);
    }
};

// Object table of the scene (analytic objects by value, grids by index) and the host image of every distinct grid.
static int build_scene_table(rm_scene_group* grp, const rm_scene* scene) {
    if (scene->objects.size() > (size_t)kMaxObjects)
        return fail(RM_ERR_UNSUPPORTED, "scene has more than " + std::to_string(kMaxObjects) + " objects");
    std::map<const Grid*, int> grid_index;
    grp->env = scene->env;
    DevScene& s = grp->table;
    s.n_objects = (int)scene->objects.size();
    s.n_grids = 0;
    for (size_t i = 0; i < scene->objects.size(); i++) {
        const Object& o = scene->objects[i];
        DevObject& d = s.obj[i];
        d.geom = o.geometry;
        d.mat = (int)o.material.kind;
        d.grid = 0;
        d.g[0] = o.origin.x; d.g[1] = o.origin.y; d.g[2] = o.origin.z;
        if (o.geometry == GEOM_SPHERE) { d.g[3] = o.radius; d.g[4] = d.g[5] = 0.0; }
        else { d.g[3] = o.normal.x; d.g[4] = o.normal.y; d.g[5] = o.normal.z; }
        d.color[0] = o.material.a.x; d.color[1] = o.material.a.y; d.color[2] = o.material.a.z;
        d.rough = o.material.p0;
        if (o.geometry == GEOM_GRID) {
            auto it = grid_index.find(o.grid.get());
            if (it == grid_index.end()) {
                if (s.n_grids >= kMaxGrids) return fail(RM_ERR_UNSUPPORTED, "scene has more than " + std::to_string(kMaxGrids) + " distinct grids");
                GridImage im;
                if (int st = prepare_grid_image(*o.grid, &im)) return st;
                grp->grids.push_back(o.grid);
                grp->images.push_back(im);
                it = grid_index.emplace(o.grid.get(), s.n_grids++).first;
            }
            d.grid = it->second;
            grp->grid_objects.push_back((int)i);
            if (d.mat == RM_MATERIAL_EMISSION) grp->emissive_grid = true;
        }
        grp->textures.push_back(o.texture);
    }
    // the uvs of a grid go up only when a textured object references it, so that an untextured scene uploads what it always did
    grp->grid_uv.assign((size_t)s.n_grids, {});
    for (size_t i = 0; i < scene->objects.size(); i++) {
        if (!scene->objects[i].texture || scene->objects[i].geometry != GEOM_GRID) continue;
        std::vector<double>& uv = grp->grid_uv[(size_t)s.obj[i].grid];
        const std::vector<rm_triangle>& tris = scene->objects[i].grid->triangles;
        if (!uv.empty() || tris.empty()) continue;
        try {
            uv.resize(tris.size() * 6);
        } catch (const std::bad_alloc&) {
            return fail(RM_ERR_OUT_OF_MEMORY, "cannot hold the uvs of a textured grid");
        }
        for (size_t k = 0; k < tris.size(); k++) {
            const rm_triangle& t = tris[k];
            double* u = uv.data() + 6 * k;
            u[0] = t.v0.uv.x; u[1] = t.v0.uv.y; u[2] = t.v1.uv.x; u[3] = t.v1.uv.y; u[4] = t.v2.uv.x; u[5] = t.v2.uv.y;
        }
    }
    return RM_OK;
}

extern "C" {

rm_scene_group* rm_scene_group_create(const rm_scene* scene, const int32_t* devices, int count) {
    if (!scene || !devices || count <= 0) { fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_group_create: bad argument"); return nullptr; }
    for (int g = 0; g < count; g++)
        if (check_device(devices[g]) != RM_OK) return nullptr;
    rm_scene_group* grp = new rm_scene_group();
    grp->devices.assign(devices, devices + count);
    grp->blocks.assign((size_t)count, {});
    grp->uploaded.assign((size_t)count, nullptr);
    const auto t0 = std::chrono::steady_clock::now();
    if (build_scene_table(grp, scene) != RM_OK) { delete grp; return nullptr; }
    grp->flatten_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return grp;
}

rm_device_scene* rm_scene_group_join(rm_scene_group* grp, int share) {
    if (!grp || share < 0 || share >= (int)grp->devices.size()) { fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_group_join: bad argument"); return nullptr; }
    const int G = (int)grp->devices.size();
    const int device = grp->devices[(size_t)share];
    rm_device_scene* ds = new rm_device_scene();
    ds->device = device;
    std::vector<void*>& mine = grp->blocks[(size_t)share];
    auto slice = [&](const GridImage& im, int j, size_t* begin, size_t* end) {
        *begin = (im.host_total * (size_t)j / (size_t)G) & ~(size_t)255;
        *end = j + 1 == G ? im.host_total : (im.host_total * (size_t)(j + 1) / (size_t)G) & ~(size_t)255;
    };
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    for (int j = 0; j < G; j++) enable_peer(device, grp->devices[(size_t)j]);      // direct NVLink copies where the hardware has them
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) {
        ds->sms = sm_count(device);
        int occ = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_traverse<false>, kTravBlock, 0) == cudaSuccess && occ > 0) ds->traverse_blocks_per_sm = occ;
        e = cudaEventCreate(&e0);
    }
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    if (e == cudaSuccess) e = cudaEventRecord(e0, 0);
    // phase 1: my slice of every image, host -> my device
    for (size_t i = 0; i < grp->images.size() && e == cudaSuccess; i++) {
        const GridImage& im = grp->images[i];
        void* dev = nullptr;
        e = visible_acquire(device, im.total, &dev);
        if (e != cudaSuccess) break;
        mine.push_back(dev);
        ds->allocations.push_back(dev);
        ds->allocation_bytes.push_back(im.total);
        size_t b, en;
        slice(im, share, &b, &en);
        if (en > b) e = cudaMemcpyAsync((char*)dev + b, im.host + b, en - b, cudaMemcpyHostToDevice, 0);
        ds->bytes += en - b;                                      // bytes that crossed the bus for this share
    }
    if (e == cudaSuccess && grp->env) {                          // the environment map: a copy per share, host -> device
        const Environment& env = *grp->env;
        const size_t bytes = env.rgba.size() * sizeof(float);
        void* dev = nullptr;
        e = visible_acquire(device, bytes, &dev);
        if (e == cudaSuccess) {
            ds->allocations.push_back(dev);
            ds->allocation_bytes.push_back(bytes);
            e = cudaMemcpyAsync(dev, env.rgba.data(), bytes, cudaMemcpyHostToDevice, 0);
            ds->bytes += bytes;
            ds->has_env = true;
            ds->env = DevEnv{(const float4*)dev, (int)env.width, (int)env.height, env.scale, env.rotation};
        }
    }
    // the colour textures and the uvs of the textured grids: a copy per share, host -> device
    auto upload = [&](const void* src, size_t bytes, void** dev) {
        cudaError_t ue = visible_acquire(device, bytes, dev);
        if (ue != cudaSuccess) return ue;
        ds->allocations.push_back(*dev);
        ds->allocation_bytes.push_back(bytes);
        ds->bytes += bytes;
        return cudaMemcpyAsync(*dev, src, bytes, cudaMemcpyHostToDevice, 0);
    };
    for (size_t i = 0; i < grp->textures.size() && e == cudaSuccess; i++) {
        if (!grp->textures[i]) continue;
        const Texture& t = *grp->textures[i];
        void* dev = nullptr;
        e = upload(t.rgba.data(), t.rgba.size() * sizeof(float), &dev);
        ds->tex.obj[i] = DevTexObject{(const float4*)dev, (int)t.width, (int)t.height, t.scale_u, t.scale_v};
        ds->has_tex = true;
    }
    for (size_t g = 0; g < grp->grid_uv.size() && e == cudaSuccess; g++) {
        if (grp->grid_uv[g].empty()) continue;
        void* dev = nullptr;
        e = upload(grp->grid_uv[g].data(), grp->grid_uv[g].size() * sizeof(double), &dev);
        ds->tex.uv[g] = (const double*)dev;
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&grp->uploaded[(size_t)share], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(grp->uploaded[(size_t)share], 0);
    bool ok = grp->barrier(0, e == cudaSuccess);
    // phase 2: the other slices from the peers that hold them (NVLink), then the per-reference spheres
    if (ok) {
        for (size_t i = 0; i < grp->images.size() && e == cudaSuccess; i++) {
            const GridImage& im = grp->images[i];
            for (int step = 1; step < G && e == cudaSuccess; step++) {
                const int j = (share + step) % G;                 // every share starts with a different peer
                size_t b, en;
                slice(im, j, &b, &en);
                if (en <= b) continue;
                e = cudaStreamWaitEvent(0, grp->uploaded[(size_t)j], 0);
                if (e == cudaSuccess)
                    e = cudaMemcpyPeerAsync((char*)mine[i] + b, device, (const char*)grp->blocks[(size_t)j][i] + b, grp->devices[(size_t)j], en - b, 0);
            }
            if (e == cudaSuccess) e = spread_spheres(im, mine[i], ds->sms, 0);
        }
        if (e == cudaSuccess) e = cudaEventRecord(e1, 0);
        if (e == cudaSuccess) e = cudaEventSynchronize(e1);
    }
    // nobody frees a block a peer may still be reading
    ok = grp->barrier(1, ok && e == cudaSuccess);
    if (ok) {
        ds->scene = grp->table;
        for (size_t i = 0; i < grp->images.size(); i++) {
            point_grid(grp->images[i], mine[i], &ds->scene.grid[i]);
            ds->tri_spheres[i] = (const float4*)((char*)mine[i] + grp->images[i].off_spht);
            ds->n_triangles[i] = grp->images[i].nt;
        }
        ds->grid_objects = grp->grid_objects;
        ds->emissive_grid = grp->emissive_grid;
        ds->keep = grp->grids;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        ds->upload_ms = grp->flatten_ms + ms;
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (!ok) {
        if (e != cudaSuccess) fail(RM_ERR_CUDA, std::string("scene upload (share ") + std::to_string(share) + "): " + cudaGetErrorString(e));
        else fail(RM_ERR_CUDA, "scene upload failed on another device of the group");
        delete ds;
        return nullptr;
    }
    return ds;
}

void rm_scene_group_destroy(rm_scene_group* grp) { delete grp; }

}  // extern "C"

namespace rm {

// Observer of the launches of one Scene::intersect pass (stage timing / launch counting).
struct LaunchHook {
    virtual void begin(int kind) = 0;
    virtual void end(int kind) = 0;
    virtual ~LaunchHook() {}
};
struct NoHook : LaunchHook {
    void begin(int) override {}
    void end(int) override {}
};

// Scene::intersect for a batch of rays: k_setup (+ k_traverse per grid object).  On return (stream
// order) `buf.hit` holds the closest hit of every ray.  `trav_count` / `cursor` are zero on entry and
// re-zeroed between grid passes.  `cover` (camera rays only): the coverage mask of the first grid object, or null (§3.7).
template <int SRC>
static int launch_intersect(rm_device_scene* ds, const RenderParams& rp, SetupArgs sa, const HitArrays& hit, double* trav, unsigned* trav_count,
                            unsigned* cursor, unsigned n_upper, unsigned depth, bool count_work, DevTotals* totals, cudaStream_t stream,
                            LaunchHook& hook, const int* cover = nullptr) {
    const unsigned setup_grid = std::max<unsigned>(1u, std::min<unsigned>((n_upper + kBlock - 1) / kBlock, (unsigned)ds->sms * 16u));
    const unsigned trav_grid = (unsigned)(ds->sms * ds->traverse_blocks_per_sm);
    sa.hit = hit;
    sa.trav = trav;
    sa.trav_count = trav_count;
    const size_t n_grid_objects = ds->grid_objects.size();
    for (size_t pass = 0; pass < std::max<size_t>(n_grid_objects, 1); pass++) {
        const int gobj = n_grid_objects ? ds->grid_objects[pass] : -1;
        sa.grid_object = gobj;
        sa.analytic = pass == 0 ? 1 : 0;
        sa.cover = pass == 0 ? cover : nullptr;
        if (pass > 0) {
            RM_CUDA(cudaMemsetAsync(trav_count, 0, sizeof(unsigned), stream));
            RM_CUDA(cudaMemsetAsync(cursor, 0, sizeof(unsigned), stream));
        }
        hook.begin(0);
        if (pass == 0) k_setup<SRC><<<setup_grid, kBlock, 0, stream>>>(ds->scene, rp, sa);
        else if (SRC == SRC_AOS) k_setup<SRC_AOS><<<setup_grid, kBlock, 0, stream>>>(ds->scene, rp, sa);
        else k_setup<SRC_QUEUE><<<setup_grid, kBlock, 0, stream>>>(ds->scene, rp, sa);   // camera rays were stored by pass 0
        hook.end(0);
        if (gobj >= 0) {
            TraverseArgs ta{};
            ta.trav = trav; ta.n_ptr = trav_count; ta.cursor = cursor; ta.hit = hit;
            ta.grid_object = gobj; ta.depth = depth; ta.totals = totals;
            const DevGrid& g = ds->scene.grid[ds->scene.obj[gobj].grid];
            hook.begin(1);
            if (count_work) k_traverse<true><<<trav_grid, kTravBlock, 0, stream>>>(g, ta);
            else k_traverse<false><<<trav_grid, kTravBlock, 0, stream>>>(g, ta);
            hook.end(1);
        }
    }
    RM_CUDA(cudaGetLastError());
    return RM_OK;
}

}  // namespace rm

// --------------------------------------------------------------------- renderer

struct rm_renderer {
    rm_device_scene* ds = nullptr;
    bool owns_scene = false;
    rm_settings settings{};
    rm_gpu_options opt{};
    int device = 0;
    int sms = 148;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    RenderParams rp{};
    Queue q[2]{};
    double* queue_mem = nullptr;
    unsigned* id_mem = nullptr;
    std::shared_ptr<rm::PixelMap> pixel_map_ref;      // shared with the other renderers of the same frame layout on this device
    unsigned* pixel_map = nullptr;
    size_t uploaded_pixel_map_bytes = 0;
    unsigned* counters = nullptr;
    size_t counter_slots = 0;
    IntersectBuffers isect;
    double* accum = nullptr;
    bool owns_accum = false;
    size_t accum_bytes = 0;
    double* moments = nullptr;                      // RM_FLAG_MOMENTS: W*H rm_vec3 running sums of squares (peers read it in place)
    double* aov = nullptr;                          // RM_FLAG_AOV: first-hit feature sums, W*H albedo rm_vec3, W*H normal rm_vec3, W*H depth
    size_t aov_bytes = 0;
    unsigned* active_map = nullptr;                 // rm_renderer_set_active_tiles: the active tiles' runs of the pixel map
    uint3* active_runs = nullptr;                   // ... and the {source, destination, length} list that gathered them
    size_t full_batch_spp = 1;                      // batch_spp for the whole share
    DevTotals* totals = nullptr;
    size_t batch_spp = 1;
    bool last_depth_shortcut = true;                // RM_FULL_LAST_BOUNCE unset: see renderer_batch_t
    bool cover_allowed = true;                      // RM_NO_COVER_MASK unset: see build_cover
    int* cover = nullptr;                           // coverage mask of the camera rays for the first grid object, null = none (§3.7)
    uint64_t launches = 0;
    double device_ms = 0.0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    struct StageEvent { cudaEvent_t a, b; unsigned kind, slot; };
    std::vector<StageEvent> stage_pending;
    std::vector<cudaEvent_t> event_pool;
    cudaEvent_t ev_rendered = nullptr, ev_reduced = nullptr;      // accumulator exchange between the renderers of one task
    double stage_ms[RM_KERNEL_KINDS][RM_STAGE_SLOTS] = {};
    uint64_t stage_launches[RM_KERNEL_KINDS][RM_STAGE_SLOTS] = {};

    ~rm_renderer() {
        cudaSetDevice(device);
        if (stream) cudaStreamSynchronize(stream);
        for (auto& p : pending) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
        for (auto& e : stage_pending) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
        for (auto& e : event_pool) cudaEventDestroy(e);
        if (ev_rendered) cudaEventDestroy(ev_rendered);
        if (ev_reduced) cudaEventDestroy(ev_reduced);
        dev_free(queue_mem); dev_free(id_mem); dev_free(rp.contrib); dev_free(counters); dev_free(totals);
        isect.release();
        if (owns_accum) visible_release(device, accum_bytes, accum);
        if (moments) visible_release(device, accum_bytes, moments);
        if (aov) visible_release(device, aov_bytes, aov);
        dev_free(active_map); dev_free(active_runs);
        dev_free(cover);
        if (owns_stream && stream) cudaStreamDestroy(stream);
        if (owns_scene) delete ds;
    }
};

namespace rm {

// Owned pixels in launch order: tiles in the reference's queue order (src/trace.rs:146-172),
// restricted to this rank's share; inside a tile, 8x4 pixel blocks so that a warp covers a compact
// screen patch (coherent primary rays walk the same grid cells).
static std::vector<unsigned> build_pixel_map(const rm_settings& s, const Share& share) {
    const size_t W = s.camera_settings.backbuffer_width, H = s.camera_settings.backbuffer_height;
    std::vector<TileRect> tiles = tile_layout(W, H, s.tile_size[0], s.tile_size[1]);
    std::vector<unsigned> map;
    map.reserve(W * H / share.tile_step() + 1024);
    for (size_t t = 0; t < tiles.size(); t++) {
        if (!share.owns_tile(t)) continue;
        const TileRect& r = tiles[t];
        for (size_t by = 0; by < r.height; by += 4)
            for (size_t bx = 0; bx < r.width; bx += 8)
                for (size_t y = by; y < std::min(by + 4, r.height); y++)
                    for (size_t x = bx; x < std::min(bx + 8, r.width); x++)
                        map.push_back((unsigned)((r.left + x) + (r.top + y) * W));
    }
    return map;
}

// The launch order of a share's pixels depends only on the frame, the tile size and the share: it is built on the host and
// uploaded once per (device, frame, tiles, owned tiles) and shared by every renderer that needs it afterwards —
// render_tiled makes a renderer per frame, and 8 MB of indices per 1080p share were 5-8 ms of every frame's start.
namespace {
struct PixelMapKey {
    int device; size_t W, H, tw, th, first, step;
    bool operator<(const PixelMapKey& o) const {
        return std::tie(device, W, H, tw, th, first, step) < std::tie(o.device, o.W, o.H, o.tw, o.th, o.first, o.step);
    }
};
std::mutex g_pixel_map_mu;
// never destroyed: its entries free device memory, which must not happen from a static destructor after the CUDA runtime is gone
std::map<PixelMapKey, std::shared_ptr<PixelMap>>& g_pixel_maps = *new std::map<PixelMapKey, std::shared_ptr<PixelMap>>();
constexpr size_t kPixelMapCacheBytes = (size_t)512 << 20;
}  // namespace

PixelMap::~PixelMap() {
    if (dev) { cudaSetDevice(device); dev_free(dev); }
}

static void pixel_map_cache_trim(size_t keep_bytes) {      // g_pixel_map_mu held
    size_t bytes = 0;
    for (auto& kv : g_pixel_maps) bytes += kv.second->n * sizeof(unsigned);
    for (auto it = g_pixel_maps.begin(); it != g_pixel_maps.end() && bytes > keep_bytes;) {
        if (it->second.use_count() == 1) { bytes -= it->second->n * sizeof(unsigned); it = g_pixel_maps.erase(it); }
        else ++it;
    }
}

static int pixel_map_for(rm_renderer* r) {
    const rm_settings& s = r->settings;
    const Share share(r->opt);
    const PixelMapKey key{r->device, s.camera_settings.backbuffer_width, s.camera_settings.backbuffer_height, s.tile_size[0], s.tile_size[1],
                          share.first_tile(), share.tile_step()};
    std::lock_guard<std::mutex> lk(g_pixel_map_mu);       // also serialises the build of a missing map between the shares of a task
    auto it = g_pixel_maps.find(key);
    if (it != g_pixel_maps.end()) { r->pixel_map_ref = it->second; return RM_OK; }
    std::vector<unsigned> map = build_pixel_map(s, share);
    auto pm = std::make_shared<PixelMap>();
    pm->device = r->device;
    pm->n = map.size();
    RM_CUDA(dev_malloc(&pm->dev, std::max<size_t>(pm->n, 1) * sizeof(unsigned)));
    if (pm->n) RM_CUDA(cudaMemcpyAsync(pm->dev, map.data(), pm->n * sizeof(unsigned), cudaMemcpyHostToDevice, r->stream));
    RM_CUDA(cudaStreamSynchronize(r->stream));
    r->uploaded_pixel_map_bytes = pm->n * sizeof(unsigned);
    pixel_map_cache_trim(kPixelMapCacheBytes);
    g_pixel_maps[key] = pm;
    r->pixel_map_ref = pm;
    return RM_OK;
}

static int renderer_init(rm_renderer* r) {
    const rm_settings& s = r->settings;
    const size_t W = s.camera_settings.backbuffer_width, H = s.camera_settings.backbuffer_height;
    if (W == 0 || H == 0 || s.tile_size[0] == 0 || s.tile_size[1] == 0) return fail(RM_ERR_INVALID_ARGUMENT, "empty backbuffer or tile size");
    if (W * H >= 0xffffffffull) return fail(RM_ERR_UNSUPPORTED, "backbuffer has 2^32 or more pixels");
    if (s.bounce_limit > 1u << 20) return fail(RM_ERR_UNSUPPORTED, "bounce_limit too large");
    if (r->opt.world_size > 1 && (r->opt.rank < 0 || r->opt.rank >= r->opt.world_size)) return fail(RM_ERR_INVALID_ARGUMENT, "rank outside world_size");
    RM_CUDA(cudaSetDevice(r->device));
    r->sms = sm_count(r->device);
    r->last_depth_shortcut = getenv("RM_FULL_LAST_BOUNCE") == nullptr;
    r->cover_allowed = getenv("RM_NO_COVER_MASK") == nullptr;
    if (r->opt.stream) r->stream = (cudaStream_t)r->opt.stream;
    else { RM_CUDA(cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking)); r->owns_stream = true; }

    Trace trace;
    if (int st = pixel_map_for(r)) return st;
    const size_t npix = r->pixel_map_ref->n;
    r->pixel_map = r->pixel_map_ref->dev;
    trace.mark("renderer_init: stream + pixel map");

    // batch: enough paths in flight to fill the machine many times over, bounded in memory
    size_t spp = r->opt.batch_spp;
    if (spp == 0) {
        // ~64 Mi paths per wavefront batch: the deep stages of a batch hold few rays, and every stage ends with the tail
        // of a persistent kernel, so bigger batches amortise both (measured at 1080p: 4 -> 16 spp +9 %, 16 -> 32 spp +1.6 %).  328 B of
        // queues per path; never more than a quarter of the free device memory.
        size_t target = (size_t)64 << 20;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) target = std::min(target, std::max<size_t>(free_b / 4 / 328, (size_t)1 << 20));
        trace.mark("renderer_init: cudaMemGetInfo");
        spp = npix ? std::max<size_t>(1, target / npix) : 1;
        spp = std::min<size_t>(spp, 64);
        // ... and never more than this share of the job renders (a rank / device of a sample-split job gets 1 / world_size of them)
        const size_t stride = Share(r->opt).sample_stride();
        spp = std::min<size_t>(spp, (std::max<size_t>(s.sample_count, 1) + stride - 1) / stride);
    }
    while (spp > 1 && spp * npix >= 0xffffffffull) spp--;
    r->batch_spp = r->full_batch_spp = spp;
    const size_t cap = std::max<size_t>(npix * spp, 32);

    RM_CUDA(dev_malloc(&r->queue_mem, cap * 9 * 2 * sizeof(double)));
    RM_CUDA(dev_malloc(&r->id_mem, cap * 2 * sizeof(unsigned)));
    for (int b = 0; b < 2; b++) {
        for (int k = 0; k < 9; k++) r->q[b].f[k] = r->queue_mem + ((size_t)b * 9 + k) * cap;
        r->q[b].id = r->id_mem + (size_t)b * cap;
    }
    if (int st = r->isect.alloc(cap)) return st;
    if (r->opt.precision != RM_PRECISION_F64 && r->opt.precision != RM_PRECISION_F32_SHADING) return fail(RM_ERR_INVALID_ARGUMENT, "unknown rm_precision");
    RenderParams& rp = r->rp;
    rp.cam = make_camera(s.camera_settings);
    rp.seed = r->opt.seed;
    rp.pixel_map = r->pixel_map;
    rp.n_pixels = (unsigned)npix;
    rp.bounce_limit = (unsigned)s.bounce_limit;
    rp.cap = (unsigned)cap;
    RM_CUDA(dev_malloc(&rp.contrib, cap * 3 * sizeof(double)));
    r->counter_slots = s.bounce_limit + 2;
    RM_CUDA(dev_malloc(&r->counters, r->counter_slots * 3 * sizeof(unsigned)));
    rp.cnt.rays = r->counters;
    rp.cnt.trav = r->counters + r->counter_slots;
    rp.cnt.cursor = r->counters + 2 * r->counter_slots;
    RM_CUDA(dev_malloc(&r->totals, sizeof(DevTotals)));
    rp.totals = r->totals;
    RM_CUDA(cudaMemsetAsync(r->totals, 0, sizeof(DevTotals), r->stream));
    r->accum_bytes = std::max<size_t>(W * H, 1) * 3 * sizeof(double);
    if (r->opt.accum_device) r->accum = (double*)r->opt.accum_device;
    else {      // not from the pool: peers read it in place
        RM_CUDA(visible_acquire(r->device, r->accum_bytes, (void**)&r->accum));
        r->owns_accum = true;
    }
    RM_CUDA(cudaMemsetAsync(r->accum, 0, W * H * 3 * sizeof(double), r->stream));
    if (r->opt.flags & RM_FLAG_MOMENTS) {
        RM_CUDA(visible_acquire(r->device, r->accum_bytes, (void**)&r->moments));
        RM_CUDA(cudaMemsetAsync(r->moments, 0, W * H * 3 * sizeof(double), r->stream));
    }
    if (r->opt.flags & RM_FLAG_AOV) {
        r->aov_bytes = std::max<size_t>(W * H, 1) * 7 * sizeof(double);
        RM_CUDA(visible_acquire(r->device, r->aov_bytes, (void**)&r->aov));
        RM_CUDA(cudaMemsetAsync(r->aov, 0, W * H * 7 * sizeof(double), r->stream));
    }
    trace.mark("renderer_init: queues, counters, accumulator allocated");
    return RM_OK;
}

// The coverage mask of the camera rays (§3.7) for the first grid object (the grid pass k_setup<SRC_CAMERA> sets up), built
// on the renderer's stream once its scene is bound: it depends only on the camera, the frame and the grid, so every batch
// and frame of the renderer reuses it.  No mask with DoF (the rays do not share an apex), under RM_FLAG_COUNT_WORK (the
// per-stage cells and tests stay comparable with the oracle's, §3.4), with RM_NO_COVER_MASK in the environment, or when the
// grid's box is not strictly in front of the camera, the error bound below is not far below a pixel, or a triangle of the
// grid cannot be projected.
static int build_cover(rm_renderer* r) {
    if (r->cover) { RM_CUDA(cudaStreamSynchronize(r->stream)); dev_free(r->cover); r->cover = nullptr; }
    const DevCamera& cam = r->rp.cam;
    if (!r->cover_allowed || cam.use_dof || (r->opt.flags & RM_FLAG_COUNT_WORK) || r->ds->grid_objects.empty()) return RM_OK;
    Trace trace;
    const int gi = r->ds->scene.obj[r->ds->grid_objects[0]].grid;
    const DevGrid& g = r->ds->scene.grid[gi];
    const size_t W = (size_t)cam.W, H = (size_t)cam.H, npx = W * H;
    // A hit Triangle::intersects accepts lies within 4e-7 * |o - v0| * diag2 of the exact triangle (the form of the bound
    // k_setup uses for t), and |o - v0| <= the distance to the farthest corner of the box: the spheres are inflated by that.
    // In pixels, a point at depth z >= zmin with |x/z|, |y/z| <= rmax moves by at most bound * (1 + rmax) / zmin.
    const double zmin = g.bmin[2] - cam.pos[2];
    double far2 = 0.0, rmax = 0.0;
    for (int k = 0; k < 8; k++) {
        const double x = (k & 1 ? g.bmax[0] : g.bmin[0]) - cam.pos[0];
        const double y = (k & 2 ? g.bmax[1] : g.bmin[1]) - cam.pos[1];
        const double z = (k & 4 ? g.bmax[2] : g.bmin[2]) - cam.pos[2];
        far2 = std::max(far2, x * x + y * y + z * z);
        rmax = std::max(rmax, std::max(std::fabs(x / z), std::fabs(y / z)));
    }
    const double inflate = 4e-7 * (std::sqrt(far2) + g.diag) * g.diag2;
    const double px_per_unit = std::max(cam.width / (2.0 * cam.tan_half * cam.aspect), cam.height / (2.0 * cam.tan_half));
    const double bound_px = inflate * (1.0 + rmax) / zmin * px_per_unit;
    if (!(zmin > 0.0) || !(bound_px < 0.25)) return RM_OK;        // NaN fails too
    int* c = nullptr;
    RM_CUDA(dev_malloc(&c, (npx + 1) * sizeof(int)));
    r->cover = c;
    RM_CUDA(cudaMemsetAsync(c, 0, (npx + 1) * sizeof(int), r->stream));
    const size_t n = r->ds->n_triangles[gi];
    if (n) {
        k_cover_rects<<<(unsigned)std::min<size_t>((n + kBlock - 1) / kBlock, (size_t)r->sms * 8), kBlock, 0, r->stream>>>(r->ds->tri_spheres[gi], n, cam,
                                                                                                                     inflate, c);
        r->launches++;
    }
    k_cover_cols<<<(unsigned)((W + kBlock - 1) / kBlock), kBlock, 0, r->stream>>>(c, (int)W, (int)H);
    k_cover_rows<<<(unsigned)((H * 32 + kBlock - 1) / kBlock), kBlock, 0, r->stream>>>(c, (int)W, (int)H);
    r->launches += 2;
    RM_CUDA(cudaGetLastError());
    int unprojectable = 0;
    RM_CUDA(cudaMemcpyAsync(&unprojectable, c + npx, sizeof(int), cudaMemcpyDeviceToHost, r->stream));
    RM_CUDA(cudaStreamSynchronize(r->stream));
    if (unprojectable) { dev_free(r->cover); r->cover = nullptr; }
    if (trace.on) {
        char line[160];
        snprintf(line, sizeof line, "renderer: coverage mask of the camera rays %s (error bound %.3g px)", r->cover ? "built" : "dropped", bound_px);
        trace.mark(line);
    }
    return RM_OK;
}

static cudaEvent_t take_event(rm_renderer* r) {
    if (!r->event_pool.empty()) { cudaEvent_t e = r->event_pool.back(); r->event_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

// Counts launches per (kernel kind, stage slot) and, with RM_FLAG_STAGE_TIMING, brackets each with events.
struct StageHook : LaunchHook {
    rm_renderer* r;
    unsigned slot;
    cudaEvent_t a = nullptr;
    StageHook(rm_renderer* r_, unsigned slot_) : r(r_), slot(slot_) {}
    void begin(int) override {
        if (r->opt.flags & RM_FLAG_STAGE_TIMING) { a = take_event(r); cudaEventRecord(a, r->stream); }
    }
    void end(int kind) override {
        r->launches++;
        r->stage_launches[kind][slot]++;
        if (a) {
            cudaEvent_t b = take_event(r);
            cudaEventRecord(b, r->stream);
            r->stage_pending.push_back({a, b, (unsigned)kind, slot});
            a = nullptr;
        }
    }
};

static const DevTex no_tex{};      // the last parameter of k_shade / k_aov for a scene without textures

// k_shade with or without the scene's environment map (env = NULL: none) and its colour textures (tex = NULL: none).  The
// LAST body shades no surface: it runs without the textures.
template <bool FIRST, int PREC, bool KEEP, bool LAST, bool ENV, bool TEX>
static void launch_shade_t(rm_renderer* r, unsigned grid, const RenderParams& rp, const Queue& qin, const Queue& qout, unsigned depth, unsigned n_first,
                           const DevEnv& env, const DevTex& tex) {
    k_shade<FIRST, PREC, KEEP, LAST, ENV, TEX><<<grid, kBlock, 0, r->stream>>>(r->ds->scene, rp, qin, qout, r->isect.hit, depth, n_first, env, tex);
}
template <bool FIRST, int PREC, bool KEEP, bool LAST>
static void launch_shade(rm_renderer* r, unsigned grid, const RenderParams& rp, const Queue& qin, const Queue& qout, unsigned depth, unsigned n_first,
                         const DevEnv* env, const DevTex* tex) {
    if (env && tex && !LAST) launch_shade_t<FIRST, PREC, KEEP, LAST, true, !LAST>(r, grid, rp, qin, qout, depth, n_first, *env, *tex);
    else if (env) launch_shade_t<FIRST, PREC, KEEP, LAST, true, false>(r, grid, rp, qin, qout, depth, n_first, *env, no_tex);
    else if (tex && !LAST) launch_shade_t<FIRST, PREC, KEEP, LAST, false, !LAST>(r, grid, rp, qin, qout, depth, n_first, DevEnv{}, *tex);
    else launch_shade_t<FIRST, PREC, KEEP, LAST, false, false>(r, grid, rp, qin, qout, depth, n_first, DevEnv{}, no_tex);
}

template <int PREC>
static int renderer_batch_t(rm_renderer* r, unsigned first_sample, unsigned n_samples, unsigned stride) {
    RenderParams rp = r->rp;
    rp.first_sample = first_sample;
    rp.sample_stride = stride;
    const unsigned n_paths = rp.n_pixels * n_samples;
    const unsigned limit = rp.bounce_limit;
    if (n_paths == 0) return RM_OK;
    const bool count = (r->opt.flags & RM_FLAG_COUNT_WORK) != 0;
    const bool keep = (r->opt.flags & RM_FLAG_KEEP_NONFINITE) != 0;
    // Drop mode at depth == bounce_limit: only whether the closest object is an emitter decides the path (k_shade<..., LAST>).
    // k_setup then skips the grids for rays whose closest analytic hit is not an emitter, unless a grid emits, or the work
    // counters must stay comparable with the reference's at every depth.  RM_FULL_LAST_BOUNCE=1 in the environment renders
    // the last depth like every other (tests compare the two; the frame is the same to the last bit).  With an environment map
    // a ray with no hit so far delivers radiance, so no traversal is skipped (k_shade<..., LAST, true> still shades the misses).
    const bool last_shade = !keep && r->last_depth_shortcut;
    const bool last_skip = last_shade && !count && !r->ds->emissive_grid && !r->ds->has_env;
    const DevEnv* env = r->ds->has_env ? &r->ds->env : nullptr;
    const DevTex* tex = r->ds->has_tex ? &r->ds->tex : nullptr;
    const unsigned persistent_grid = (unsigned)r->sms * 8u;
    RM_CUDA(cudaMemsetAsync(r->counters, 0, r->counter_slots * 3 * sizeof(unsigned), r->stream));
    if (limit == 0) RM_CUDA(cudaMemsetAsync(rp.contrib, 0, (size_t)rp.cap * 3 * sizeof(double), r->stream));   // trace() returns 0 at depth 1 > 0
    for (unsigned depth = 1; depth <= limit; depth++) {
        StageHook hook(r, stage_slot(depth));
        const Queue& qin = r->q[(depth - 1) & 1];     // rays of this depth (depth 1: written by k_setup<SRC_CAMERA>)
        const Queue& qout = r->q[depth & 1];
        SetupArgs sa{};
        for (int k = 0; k < 6; k++) sa.q[k] = qin.f[k];
        // the feature buffers need the closest hit of every camera ray, so depth 1 never skips a grid for them
        sa.emitters_only = last_skip && depth == limit && !(depth == 1 && r->aov) ? 1 : 0;
        int st;
        if (depth == 1) {
            sa.n_ptr = nullptr; sa.n_direct = n_paths;
            st = launch_intersect<SRC_CAMERA>(r->ds, rp, sa, r->isect.hit, r->isect.trav, &rp.cnt.trav[depth], &rp.cnt.cursor[depth], n_paths, depth, count,
                                              r->totals, r->stream, hook, r->cover);
        } else {
            sa.n_ptr = &rp.cnt.rays[depth - 1]; sa.n_direct = 0;
            st = launch_intersect<SRC_QUEUE>(r->ds, rp, sa, r->isect.hit, r->isect.trav, &rp.cnt.trav[depth], &rp.cnt.cursor[depth], persistent_grid * kBlock,
                                             depth, count, r->totals, r->stream, hook);
        }
        if (st != RM_OK) return st;
        if (depth == 1 && r->aov) {     // before k_shade: the next depth's k_setup overwrites the hit records
            const size_t W = r->settings.camera_settings.backbuffer_width, H = r->settings.camera_settings.backbuffer_height;
            const unsigned blocks = (rp.n_pixels + kBlock - 1) / kBlock;
            if (tex) k_aov<true><<<blocks, kBlock, 0, r->stream>>>(r->ds->scene, rp, qin, r->isect.hit, n_samples, W * H, r->aov, *tex);
            else k_aov<false><<<blocks, kBlock, 0, r->stream>>>(r->ds->scene, rp, qin, r->isect.hit, n_samples, W * H, r->aov, no_tex);
            r->launches++;
        }
        hook.begin(2);
        const bool last = last_shade && depth == limit;
        if (depth == 1) {
            const unsigned grid = std::min<unsigned>((n_paths + kBlock - 1) / kBlock, persistent_grid * 4u);
            if (keep) launch_shade<true, PREC, true, false>(r, grid, rp, qin, qout, depth, n_paths, env, tex);
            else if (last) launch_shade<true, PREC, false, true>(r, grid, rp, qin, qout, depth, n_paths, env, tex);
            else launch_shade<true, PREC, false, false>(r, grid, rp, qin, qout, depth, n_paths, env, tex);
        } else {
            if (keep) launch_shade<false, PREC, true, false>(r, persistent_grid, rp, qin, qout, depth, 0u, env, tex);
            else if (last) launch_shade<false, PREC, false, true>(r, persistent_grid, rp, qin, qout, depth, 0u, env, tex);
            else launch_shade<false, PREC, false, false>(r, persistent_grid, rp, qin, qout, depth, 0u, env, tex);
        }
        hook.end(2);
    }
    {
        StageHook hook(r, 0);
        hook.begin(3);
        const unsigned blocks = (rp.n_pixels + kBlock - 1) / kBlock;
        if (r->moments) k_accumulate<true><<<blocks, kBlock, 0, r->stream>>>(rp, r->accum, n_samples, keep ? 1u : 0u, r->moments);
        else k_accumulate<false><<<blocks, kBlock, 0, r->stream>>>(rp, r->accum, n_samples, keep ? 1u : 0u, nullptr);
        hook.end(3);
    }
    RM_CUDA(cudaGetLastError());
    return RM_OK;
}

static int renderer_batch(rm_renderer* r, unsigned first_sample, unsigned n_samples, unsigned stride) {
    if (r->opt.precision == RM_PRECISION_F32_SHADING) return renderer_batch_t<RM_PRECISION_F32_SHADING>(r, first_sample, n_samples, stride);
    return renderer_batch_t<RM_PRECISION_F64>(r, first_sample, n_samples, stride);
}

static void harvest_events(rm_renderer* r) {
    for (auto& p : r->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.first, p.second) == cudaSuccess) r->device_ms += ms;
        cudaEventDestroy(p.first);
        cudaEventDestroy(p.second);
    }
    r->pending.clear();
    for (auto& e : r->stage_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) r->stage_ms[e.kind][e.slot] += ms;
        r->event_pool.push_back(e.a);
        r->event_pool.push_back(e.b);
    }
    r->stage_pending.clear();
}

}  // namespace rm

namespace rm {

__global__ void __launch_bounds__(256) k_add(double* __restrict__ total, const double* __restrict__ part, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) total[i] += part[i];
}

// The accumulator exchange of a multi-device task as ONE pass: elements [begin, end) of the frame summed over all the
// devices' accumulators (read in place over NVLink peer mappings, in device order — the association of a sequential
// "total += part" chain, so the frame does not depend on which device sums which slice) and written straight into the
// pinned host frame the tile messages are sliced from.  Every device runs this on its own slice: reduce-scatter over
// peer memory + the D2H of the result over that device's own PCIe link, no staging copy, no gather onto one device.
struct SharePointers {
    const double* acc[kMaxShares];
    int count;
};
// `mean` (optional): the finalize fused in — tile.data[..] / tile.sample_count as f64 (src/trace.rs:95), so that await() only copies.
__global__ void __launch_bounds__(256) k_reduce_slice(const __grid_constant__ SharePointers p, double* __restrict__ out, double* __restrict__ mean,
                                                        double divisor, size_t begin, size_t end) {
    for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += (size_t)gridDim.x * blockDim.x) {
        double s = p.acc[0][i];
        for (int j = 1; j < p.count; j++) s += p.acc[j][i];
        out[i] = s;
        if (mean) mean[i] = s / divisor;
    }
}

// every device of the shares reads every other's memory in place, and one kernel parameter block takes all their pointers
static bool peers_mapped(rm_renderer* const* rs, int count) {
    if (count > kMaxShares) return false;
    for (int g = 0; g < count; g++)
        for (int j = 0; j < count; j++)
            if (!enable_peer(rs[g]->device, rs[j]->device)) return false;
    return true;
}

// The staged exchange, for shares whose devices cannot all read each other's memory: `total` = the n doubles at `buf` of every
// renderer summed in renderer order, with a peer copy into `part` + k_add per renderer on the first renderer's stream (both
// buffers on its device).  Everything the other renderers enqueued is complete on entry.
static cudaError_t stage_sum(rm_renderer* const* rs, int count, double* rm_renderer::*buf, double* total, double* part, size_t n) {
    rm_renderer* r0 = rs[0];
    cudaError_t e = cudaMemcpyAsync(total, r0->*buf, n * sizeof(double), cudaMemcpyDeviceToDevice, r0->stream);
    const unsigned blocks = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)r0->sms * 16);
    for (int g = 1; g < count && e == cudaSuccess; g++) {
        e = cudaMemcpyPeerAsync(part, r0->device, rs[g]->*buf, rs[g]->device, n * sizeof(double), r0->stream);
        if (e == cudaSuccess) { k_add<<<blocks, 256, 0, r0->stream>>>(total, part, n); r0->launches++; e = cudaGetLastError(); }
    }
    return e;
}

// Fallback when the destination is pageable memory (pinning failed) or k_reduce_slice cannot read every accumulator in place:
// the staged sum, then one D2H copy.
static int reduce_gather_to_host(rm_renderer* const* rs, int count, rm_vec3* out) {
    rm_renderer* r0 = rs[0];
    const size_t n = r0->settings.camera_settings.backbuffer_width * r0->settings.camera_settings.backbuffer_height * 3;
    for (int g = 1; g < count; g++) {            // everything the peers rendered must be complete before it is copied
        RM_CUDA(cudaSetDevice(rs[g]->device));
        RM_CUDA(cudaStreamSynchronize(rs[g]->stream));
    }
    RM_CUDA(cudaSetDevice(r0->device));
    double *total = nullptr, *part = nullptr;
    cudaError_t e = dev_malloc(&total, n * sizeof(double));
    if (e == cudaSuccess) e = dev_malloc(&part, n * sizeof(double));
    if (e == cudaSuccess) e = stage_sum(rs, count, &rm_renderer::accum, total, part, n);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, total, n * sizeof(double), cudaMemcpyDeviceToHost, r0->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(r0->stream);
    dev_free(total);
    dev_free(part);
    if (e != cudaSuccess) return fail(RM_ERR_CUDA, std::string("accumulator reduce: ") + cudaGetErrorString(e));
    return RM_OK;
}

int reduce_accumulators_to_host(rm_renderer* const* rs, int count, rm_vec3* out, bool out_is_pinned, rm_vec3* mean_pinned, double divisor, bool* mean_written) {
    if (mean_written) *mean_written = false;
    if (count <= 0 || !rs || !out) return fail(RM_ERR_INVALID_ARGUMENT, "reduce_accumulators_to_host: bad argument");
    rm_renderer* r0 = rs[0];
    const size_t n = r0->settings.camera_settings.backbuffer_width * r0->settings.camera_settings.backbuffer_height * 3;
    if (count == 1) {
        RM_CUDA(cudaSetDevice(r0->device));
        RM_CUDA(cudaMemcpyAsync(out, r0->accum, n * sizeof(double), cudaMemcpyDeviceToHost, r0->stream));
        RM_CUDA(cudaStreamSynchronize(r0->stream));
        return RM_OK;
    }
    if (!out_is_pinned || !peers_mapped(rs, count)) return reduce_gather_to_host(rs, count, out);
    // the frame as the devices see it (the same address under unified addressing)
    double *out_dev = nullptr, *mean_dev = nullptr;
    RM_CUDA(cudaSetDevice(r0->device));
    if (cudaHostGetDevicePointer((void**)&out_dev, (void*)out, 0) != cudaSuccess) { cudaGetLastError(); return reduce_gather_to_host(rs, count, out); }
    if (mean_pinned && cudaHostGetDevicePointer((void**)&mean_dev, (void*)mean_pinned, 0) != cudaSuccess) { cudaGetLastError(); mean_dev = nullptr; }
    SharePointers p{};
    p.count = count;
    for (int g = 0; g < count; g++) p.acc[g] = rs[g]->accum;
    for (int g = 0; g < count; g++) {
        RM_CUDA(cudaSetDevice(rs[g]->device));
        if (!rs[g]->ev_rendered) RM_CUDA(cudaEventCreateWithFlags(&rs[g]->ev_rendered, cudaEventDisableTiming));
        if (!rs[g]->ev_reduced) RM_CUDA(cudaEventCreateWithFlags(&rs[g]->ev_reduced, cudaEventDisableTiming));
        RM_CUDA(cudaEventRecord(rs[g]->ev_rendered, rs[g]->stream));
    }
    for (int g = 0; g < count; g++) {
        rm_renderer* r = rs[g];
        RM_CUDA(cudaSetDevice(r->device));
        for (int j = 0; j < count; j++)
            if (j != g) RM_CUDA(cudaStreamWaitEvent(r->stream, rs[j]->ev_rendered, 0));      // everything the peers rendered is complete
        const size_t begin = (n * (size_t)g / (size_t)count) & ~(size_t)31, end = g + 1 == count ? n : (n * (size_t)(g + 1) / (size_t)count) & ~(size_t)31;
        if (end > begin) {
            const unsigned blocks = (unsigned)std::min<size_t>((end - begin + 255) / 256, (size_t)r->sms * 8);
            k_reduce_slice<<<blocks, 256, 0, r->stream>>>(p, out_dev, mean_dev, divisor, begin, end);
            r->launches++;
        }
        RM_CUDA(cudaGetLastError());
        RM_CUDA(cudaEventRecord(r->ev_reduced, r->stream));
    }
    // no device goes on accumulating before every peer has read its sums (the exchange is non-destructive: rendering continues)
    for (int g = 0; g < count; g++) {
        RM_CUDA(cudaSetDevice(rs[g]->device));
        for (int j = 0; j < count; j++)
            if (j != g) RM_CUDA(cudaStreamWaitEvent(rs[g]->stream, rs[j]->ev_reduced, 0));
    }
    for (int g = 0; g < count; g++) {
        cudaError_t e = cudaEventSynchronize(rs[g]->ev_reduced);
        if (e != cudaSuccess) return fail(RM_ERR_CUDA, std::string("accumulator exchange: ") + cudaGetErrorString(e));
    }
    if (mean_written) *mean_written = mean_dev != nullptr;
    return RM_OK;
}

// E_t (include/raymond.h) of tiles first, first + step, ... of the layout after `n` samples, from the sums listed in `sm`,
// on r's stream, into out_dev[tile].
static int launch_tile_error(rm_renderer* r, const ShareMoments& sm, double* out_dev, size_t n_tiles, size_t first, size_t step, double n) {
    if (first >= n_tiles) return RM_OK;
    const rm_settings& s = r->settings;
    const size_t W = s.camera_settings.backbuffer_width, H = s.camera_settings.backbuffer_height;
    const unsigned blocks = (unsigned)((n_tiles - first + step - 1) / step);
    RM_CUDA(cudaSetDevice(r->device));
    k_tile_error<<<blocks, kTileErrorBlock, 0, r->stream>>>(sm, out_dev, (unsigned)W, (unsigned)H, (unsigned)std::min(s.tile_size[0], W),
                                                             (unsigned)std::min(s.tile_size[1], H), (unsigned)first, (unsigned)step, n);
    r->launches++;
    RM_CUDA(cudaGetLastError());
    return RM_OK;
}

int tile_errors_to_host(rm_renderer* const* rs, int count, size_t n, double* out_pinned, size_t n_tiles, size_t first, size_t step) {
    if (count <= 0 || !rs || !out_pinned) return fail(RM_ERR_INVALID_ARGUMENT, "tile_errors_to_host: bad argument");
    for (int g = 0; g < count; g++) {
        if (!rs[g]->moments) return fail(RM_ERR_STATE, "tile errors need RM_FLAG_MOMENTS");
        RM_CUDA(cudaSetDevice(rs[g]->device));
        RM_CUDA(cudaStreamSynchronize(rs[g]->stream));      // every share's sums are complete before any device reads them
    }
    double* out_dev = nullptr;
    RM_CUDA(cudaHostGetDevicePointer((void**)&out_dev, (void*)out_pinned, 0));
    rm_renderer* r0 = rs[0];
    if (peers_mapped(rs, count)) {
        // every device sums the shares in place (peer reads, in device order) for its tiles
        ShareMoments sm{};
        sm.count = count;
        for (int g = 0; g < count; g++) { sm.acc[g] = rs[g]->accum; sm.mom[g] = rs[g]->moments; }
        for (int g = 0; g < count; g++)
            if (int st = launch_tile_error(rs[g], sm, out_dev, n_tiles, first + (size_t)g * step, (size_t)count * step, (double)n)) return st;
        for (int g = 0; g < count; g++) {
            RM_CUDA(cudaSetDevice(rs[g]->device));
            RM_CUDA(cudaStreamSynchronize(rs[g]->stream));
        }
        return RM_OK;
    }
    // no peer mapping: S and Q staged onto the first device
    const size_t len = r0->settings.camera_settings.backbuffer_width * r0->settings.camera_settings.backbuffer_height * 3;
    RM_CUDA(cudaSetDevice(r0->device));
    double *S = nullptr, *Q = nullptr, *part = nullptr;
    cudaError_t e = dev_malloc(&S, len * sizeof(double));
    if (e == cudaSuccess) e = dev_malloc(&Q, len * sizeof(double));
    if (e == cudaSuccess) e = dev_malloc(&part, len * sizeof(double));
    if (e == cudaSuccess) e = stage_sum(rs, count, &rm_renderer::accum, S, part, len);
    if (e == cudaSuccess) e = stage_sum(rs, count, &rm_renderer::moments, Q, part, len);
    int st = RM_OK;
    if (e == cudaSuccess) {
        ShareMoments sm{};
        sm.count = 1;
        sm.acc[0] = S;
        sm.mom[0] = Q;
        st = launch_tile_error(r0, sm, out_dev, n_tiles, first, step, (double)n);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(r0->stream);
    dev_free(S); dev_free(Q); dev_free(part);
    if (e != cudaSuccess) return fail(RM_ERR_CUDA, std::string("tile errors: ") + cudaGetErrorString(e));
    return st;
}

// The sliced filter: stage 0 reduces and packs every share's rows, stage i + 1 is pass i.  A stage reads what the previous one
// wrote, in place on every peer, and overwrites the colour plane the previous one read, so every share's stage waits for every
// share's previous stage (cross-device events, as the accumulator exchange orders itself).
static int denoise_sliced(rm_renderer* const* rs, int count, size_t n, const rm_denoise_settings& s, rm_vec3* out_dev) {
    const size_t W = rs[0]->settings.camera_settings.backbuffer_width, H = rs[0]->settings.camera_settings.backbuffer_height;
    DenoiseSlices d{};
    d.count = count;
    std::vector<size_t> bytes(count);
    cudaError_t e = cudaSuccess;
    for (int g = 0; g < count; g++) {
        d.sums[g] = rs[g]->accum;
        d.moments[g] = rs[g]->moments;
        d.aov[g] = rs[g]->aov;
    }
    // not from the pool: peers read the packed rows in place
    for (int g = 0; g < count && e == cudaSuccess; g++) {
        bytes[g] = std::max<size_t>((slice_begin(H, g + 1, count) - slice_begin(H, g, count)) * W, 1) * 4 * sizeof(float4);
        e = cudaSetDevice(rs[g]->device);
        if (e == cudaSuccess) e = visible_acquire(rs[g]->device, bytes[g], &d.packed[g]);
    }
    for (int g = 0; g < count && e == cudaSuccess; g++) {       // the sums every share reads are complete
        e = cudaSetDevice(rs[g]->device);
        if (e == cudaSuccess && !rs[g]->ev_rendered) e = cudaEventCreateWithFlags(&rs[g]->ev_rendered, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventRecord(rs[g]->ev_rendered, rs[g]->stream);
    }
    for (uint32_t stage = 0; stage <= s.iterations && e == cudaSuccess; stage++) {
        // all waits of a stage are enqueued before any share records the stage's event
        for (int g = 0; g < count && e == cudaSuccess; g++) {
            e = cudaSetDevice(rs[g]->device);
            for (int j = 0; j < count && e == cudaSuccess; j++)
                if (j != g) e = cudaStreamWaitEvent(rs[g]->stream, rs[j]->ev_rendered, 0);
        }
        for (int g = 0; g < count && e == cudaSuccess; g++) {
            rm_renderer* r = rs[g];
            e = cudaSetDevice(r->device);
            if (e == cudaSuccess)
                e = (cudaError_t)(stage == 0 ? denoise_reduce_slice(d, g, W, H, (double)n, r->stream)
                                             : denoise_pass_slice(d, g, W, H, stage - 1, s, stage == s.iterations ? out_dev : nullptr, r->stream));
            if (e == cudaSuccess && slice_begin(H, g + 1, count) > slice_begin(H, g, count)) r->launches++;
            if (e == cudaSuccess) e = cudaEventRecord(r->ev_rendered, r->stream);
        }
    }
    for (int g = 0; g < count; g++) {           // before the packed rows go back to the cache
        cudaSetDevice(rs[g]->device);
        const cudaError_t done = cudaStreamSynchronize(rs[g]->stream);
        if (e == cudaSuccess) e = done;
    }
    for (int g = 0; g < count; g++) visible_release(rs[g]->device, bytes[g], d.packed[g]);
    if (e != cudaSuccess) return fail(RM_ERR_CUDA, std::string("sliced denoiser: ") + cudaGetErrorString(e));
    return RM_OK;
}

int denoise_shares_to_host(rm_renderer* const* rs, int count, size_t n, const rm_denoise_settings& s, rm_vec3* out_pinned) {
    if (count <= 0 || !rs || !out_pinned) return fail(RM_ERR_INVALID_ARGUMENT, "denoise_shares_to_host: bad argument");
    for (int g = 0; g < count; g++)
        if (!rs[g]->aov || !rs[g]->moments) return fail(RM_ERR_STATE, "the denoiser needs RM_FLAG_AOV and RM_FLAG_MOMENTS");
    rm_renderer* r0 = rs[0];
    const size_t W = r0->settings.camera_settings.backbuffer_width, H = r0->settings.camera_settings.backbuffer_height, np = W * H;
    RM_CUDA(cudaSetDevice(r0->device));
    rm_vec3* out_dev = nullptr;      // the frame as the devices see it (the same address under unified addressing)
    RM_CUDA(cudaHostGetDevicePointer((void**)&out_dev, (void*)out_pinned, 0));
    if (count == 1) {
        const int st = denoise_to_host(r0->accum, r0->moments, r0->aov, W, H, (double)n, s, out_dev, r0->stream);
        if (st == RM_OK) r0->launches += 1 + s.iterations;
        return st;
    }
    if (peers_mapped(rs, count)) return denoise_sliced(rs, count, n, s, out_dev);
    // no peer mapping (or more shares than one kernel takes): S, Q and the features staged onto the first device
    for (int g = 0; g < count; g++) {
        RM_CUDA(cudaSetDevice(rs[g]->device));
        RM_CUDA(cudaStreamSynchronize(rs[g]->stream));
    }
    RM_CUDA(cudaSetDevice(r0->device));
    double *S = nullptr, *Q = nullptr, *A = nullptr, *part = nullptr;
    cudaError_t e = dev_malloc(&S, np * 3 * sizeof(double));
    if (e == cudaSuccess) e = dev_malloc(&Q, np * 3 * sizeof(double));
    if (e == cudaSuccess) e = dev_malloc(&A, np * 7 * sizeof(double));
    if (e == cudaSuccess) e = dev_malloc(&part, np * 7 * sizeof(double));
    if (e == cudaSuccess) e = stage_sum(rs, count, &rm_renderer::accum, S, part, np * 3);
    if (e == cudaSuccess) e = stage_sum(rs, count, &rm_renderer::moments, Q, part, np * 3);
    if (e == cudaSuccess) e = stage_sum(rs, count, &rm_renderer::aov, A, part, np * 7);
    int st = RM_OK;
    if (e == cudaSuccess) {
        st = denoise_to_host(S, Q, A, W, H, (double)n, s, out_dev, r0->stream);
        if (st == RM_OK) r0->launches += 1 + s.iterations;
    }
    const cudaError_t done = cudaStreamSynchronize(r0->stream);      // before the staging buffers go back to the pool
    if (e == cudaSuccess) e = done;
    dev_free(S); dev_free(Q); dev_free(A); dev_free(part);
    if (e != cudaSuccess) return fail(RM_ERR_CUDA, std::string("staged denoiser: ") + cudaGetErrorString(e));
    return st;
}

}  // namespace rm

// ===================================================================== C ABI (device level)

extern "C" {

rm_device_scene* rm_device_scene_create(const rm_scene* scene, int device) {
    if (!scene) { fail(RM_ERR_INVALID_ARGUMENT, "rm_device_scene_create: null scene"); return nullptr; }
    rm_scene_group* grp = rm_scene_group_create(scene, &device, 1);
    if (!grp) return nullptr;
    rm_device_scene* ds = rm_scene_group_join(grp, 0);
    rm_scene_group_destroy(grp);
    return ds;
}

void rm_device_scene_destroy(rm_device_scene* ds) { delete ds; }

rm_device_scene* rm_renderer_device_scene(rm_renderer* r) { return r ? r->ds : nullptr; }

int rm_device_scene_intersect(rm_device_scene* ds, const rm_ray* rays, size_t count, int64_t* obj, uint64_t* sub, double* distance, void* stream_) {
    if (!ds || (!rays && count)) return fail(RM_ERR_INVALID_ARGUMENT, "rm_device_scene_intersect: null argument");
    if (count == 0) return RM_OK;
    if (count >= 0xffffffffull) return fail(RM_ERR_UNSUPPORTED, "more than 2^32 - 1 rays in one call");
    cudaStream_t stream = (cudaStream_t)stream_;
    RM_CUDA(cudaSetDevice(ds->device));
    std::lock_guard<std::mutex> lk(ds->query_mu);
    if (ds->query.cap < count) {
        RM_CUDA(cudaDeviceSynchronize());   // earlier queries may still use the old scratch
        ds->query.release();
        if (int st = ds->query.alloc(count)) return st;
    }
    if (!ds->query_counters) RM_CUDA(dev_malloc(&ds->query_counters, 2 * sizeof(unsigned)));
    // one scratch set per device scene: calls on different streams are ordered one after the other on the device
    if (!ds->query_done) RM_CUDA(cudaEventCreateWithFlags(&ds->query_done, cudaEventDisableTiming));
    else RM_CUDA(cudaStreamWaitEvent(stream, ds->query_done, 0));
    RM_CUDA(cudaMemsetAsync(ds->query_counters, 0, 2 * sizeof(unsigned), stream));
    RenderParams rp{};
    SetupArgs sa{};
    sa.aos = rays;
    sa.n_ptr = nullptr;
    sa.n_direct = (unsigned)count;
    NoHook hook;
    if (int st = launch_intersect<SRC_AOS>(ds, rp, sa, ds->query.hit, ds->query.trav, ds->query_counters, ds->query_counters + 1, (unsigned)count, 1u, false,
                                           nullptr, stream, hook))
        return st;
    const size_t blocks = std::min<size_t>((count + kBlock - 1) / kBlock, (size_t)ds->sms * 32);
    k_export_hits<<<(unsigned)blocks, kBlock, 0, stream>>>(ds->query.hit, count, (long long*)obj, (unsigned long long*)sub, distance);
    RM_CUDA(cudaGetLastError());
    RM_CUDA(cudaEventRecord(ds->query_done, stream));
    return RM_OK;
}

int rm_primary_rays_device(const rm_camera_settings* camera, int device, rm_ray* rays, void* stream) {
    if (!camera || !rays) return fail(RM_ERR_INVALID_ARGUMENT, "rm_primary_rays_device: null argument");
    RM_CUDA(cudaSetDevice(device));
    DevCamera cam = make_camera(*camera);
    const size_t n = (size_t)cam.W * cam.H;
    if (n == 0) return RM_OK;
    const size_t blocks = std::min<size_t>((n + kBlock - 1) / kBlock, (size_t)sm_count(device) * 32);
    k_primary_rays<<<(unsigned)blocks, kBlock, 0, (cudaStream_t)stream>>>(cam, rays);
    RM_CUDA(cudaGetLastError());
    return RM_OK;
}

int rm_scene_intersect(const rm_scene* scene, int device, const rm_ray* rays, size_t count, int64_t* obj, uint64_t* sub, double* distance) {
    if (!scene || (!rays && count)) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_intersect: null argument");
    rm_device_scene* ds = rm_device_scene_create(scene, device);
    if (!ds) return rm_last_status();
    int st = RM_OK;
    rm_ray* d_rays = nullptr; int64_t* d_obj = nullptr; uint64_t* d_sub = nullptr; double* d_t = nullptr;
    auto cleanup = [&]() { dev_free(d_rays); dev_free(d_obj); dev_free(d_sub); dev_free(d_t); delete ds; };
#define RM_TRY(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { st = fail(RM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); cleanup(); return st; } } while (0)
    if (count) {
        RM_TRY(dev_malloc(&d_rays, count * sizeof(rm_ray)));
        RM_TRY(dev_malloc(&d_obj, count * sizeof(int64_t)));
        RM_TRY(dev_malloc(&d_sub, count * sizeof(uint64_t)));
        RM_TRY(dev_malloc(&d_t, count * sizeof(double)));
        RM_TRY(cudaMemcpy(d_rays, rays, count * sizeof(rm_ray), cudaMemcpyHostToDevice));
        if (distance) RM_TRY(cudaMemcpy(d_t, distance, count * sizeof(double), cudaMemcpyHostToDevice));   // misses leave it untouched
        st = rm_device_scene_intersect(ds, d_rays, count, d_obj, d_sub, d_t, nullptr);
        if (st == RM_OK) {
            RM_TRY(cudaDeviceSynchronize());
            if (obj) RM_TRY(cudaMemcpy(obj, d_obj, count * sizeof(int64_t), cudaMemcpyDeviceToHost));
            if (sub) RM_TRY(cudaMemcpy(sub, d_sub, count * sizeof(uint64_t), cudaMemcpyDeviceToHost));
            if (distance) RM_TRY(cudaMemcpy(distance, d_t, count * sizeof(double), cudaMemcpyDeviceToHost));
        }
    }
#undef RM_TRY
    cleanup();
    return st;
}

/* A renderer without a scene yet: stream, pixel map, wavefront queues, accumulator on options->device.  Lets the shares of a
 * multi-device task set themselves up while the scene is still being uploaded and gathered. */
rm_renderer* rm_renderer_create_unbound(const rm_settings* settings, const rm_gpu_options* options) {
    if (!settings) { fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_create_unbound: null argument"); return nullptr; }
    if (validate_camera(settings->camera_settings, "rm_renderer_create_unbound") != RM_OK) return nullptr;
    rm_renderer* r = new rm_renderer();
    r->settings = *settings;
    if (options) r->opt = *options;
    r->opt.device_list = nullptr;
    r->device = r->opt.device;
    if (check_device(r->device) != RM_OK || renderer_init(r) != RM_OK) { delete r; return nullptr; }
    return r;
}

int rm_renderer_bind_scene(rm_renderer* r, rm_device_scene* ds, int owning) {
    if (!r || !ds) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_bind_scene: null argument");
    if (ds->device != r->device) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_bind_scene: the scene lives on another device");
    r->ds = ds;
    r->owns_scene = owning != 0;
    RM_CUDA(cudaSetDevice(r->device));
    return build_cover(r);
}

// The coverage mask of the camera rays (§3.7), as W*H ints 0 / 1 (row-major); RM_ERR_STATE when the renderer has none.
int rm_renderer_coverage(rm_renderer* r, int32_t* out_host) {
    if (!r || !out_host) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_coverage: null argument");
    const int* c = r->cover;
    if (!c) return fail(RM_ERR_STATE, "rm_renderer_coverage: the renderer's camera rays have no coverage mask");
    RM_CUDA(cudaSetDevice(r->device));
    RM_CUDA(cudaMemcpyAsync(out_host, c, (size_t)r->rp.cam.W * r->rp.cam.H * sizeof(int), cudaMemcpyDeviceToHost, r->stream));
    RM_CUDA(cudaStreamSynchronize(r->stream));
    return RM_OK;
}

rm_renderer* rm_renderer_create_on(rm_device_scene* ds, const rm_settings* settings, const rm_gpu_options* options) {
    if (!ds || !settings) { fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_create_on: null argument"); return nullptr; }
    rm_gpu_options o{};
    if (options) o = *options;
    o.device = ds->device;
    rm_renderer* r = rm_renderer_create_unbound(settings, &o);
    if (r) rm_renderer_bind_scene(r, ds, 0);
    return r;
}

rm_renderer* rm_renderer_create(const rm_scene* scene, const rm_settings* settings, const rm_gpu_options* options) {
    if (!scene || !settings) { fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_create: null argument"); return nullptr; }
    if (validate_camera(settings->camera_settings, "rm_renderer_create") != RM_OK) return nullptr;   // before the scene upload
    rm_device_scene* ds = rm_device_scene_create(scene, options ? options->device : 0);
    if (!ds) return nullptr;
    rm_renderer* r = rm_renderer_create_on(ds, settings, options);
    if (!r) { delete ds; return nullptr; }
    r->owns_scene = true;
    return r;
}

int rm_renderer_render(rm_renderer* r, size_t first_sample, size_t count, size_t stride) {
    if (!r) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_render: null renderer");
    if (!r->ds) return fail(RM_ERR_STATE, "rm_renderer_render: no scene bound to the renderer");
    if (stride == 0) stride = 1;
    if (first_sample + count * stride >= 0xffffffffull) return fail(RM_ERR_UNSUPPORTED, "sample index beyond 2^32");
    RM_CUDA(cudaSetDevice(r->device));
    cudaEvent_t e0, e1;
    RM_CUDA(cudaEventCreate(&e0));
    RM_CUDA(cudaEventCreate(&e1));
    RM_CUDA(cudaEventRecord(e0, r->stream));
    size_t done = 0;
    int st = RM_OK;
    while (done < count && st == RM_OK) {
        const size_t nb = std::min(r->batch_spp, count - done);
        st = renderer_batch(r, (unsigned)(first_sample + done * stride), (unsigned)nb, (unsigned)stride);
        done += nb;
    }
    cudaEventRecord(e1, r->stream);
    r->pending.emplace_back(e0, e1);
    return st;
}

void* rm_renderer_accum_device(rm_renderer* r) { return r ? r->accum : nullptr; }

int rm_renderer_clear(rm_renderer* r) {
    if (!r) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_clear: null renderer");
    RM_CUDA(cudaSetDevice(r->device));
    const size_t n = r->settings.camera_settings.backbuffer_width * r->settings.camera_settings.backbuffer_height * 3;
    RM_CUDA(cudaMemsetAsync(r->accum, 0, n * sizeof(double), r->stream));   // statistics stay cumulative
    if (r->moments) RM_CUDA(cudaMemsetAsync(r->moments, 0, n * sizeof(double), r->stream));
    if (r->aov) RM_CUDA(cudaMemsetAsync(r->aov, 0, n / 3 * 7 * sizeof(double), r->stream));
    return RM_OK;
}

int rm_renderer_sync(rm_renderer* r) {
    if (!r) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_sync: null renderer");
    RM_CUDA(cudaSetDevice(r->device));
    RM_CUDA(cudaStreamSynchronize(r->stream));
    harvest_events(r);
    return RM_OK;
}

// The accumulator to (pageable) caller memory: D2H at link speed into a cached pinned block, then a few host threads move
// it on, dividing by `divisor` on the way (tile.data[..] / tile.sample_count as f64, src/trace.rs:95) when it is not 0.
// `source` / `count`: another W*H-sized buffer of `count` doubles (default: the accumulator, W*H rm_vec3).
static int read_accumulator(rm_renderer* r, void* out_host, double divisor, const double* source = nullptr, size_t count = 0) {
    RM_CUDA(cudaSetDevice(r->device));
    const size_t n = count ? count : r->settings.camera_settings.backbuffer_width * r->settings.camera_settings.backbuffer_height * 3;
    double* const out = (double*)out_host;
    double* pin = (double*)pinned_acquire(std::max<size_t>(n, 1) * sizeof(double));
    cudaError_t e = cudaMemcpyAsync(pin ? pin : out, source ? source : r->accum, n * sizeof(double), cudaMemcpyDeviceToHost, r->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(r->stream);
    if (e != cudaSuccess) {
        pinned_release(pin);
        return fail(RM_ERR_CUDA, std::string("D2H of the accumulator: ") + cudaGetErrorString(e));
    }
    harvest_events(r);
    const double* src = pin ? pin : out;
    auto rows = [&](size_t lo, size_t hi) {
        if (divisor != 0.0) for (size_t i = lo; i < hi; i++) out[i] = src[i] / divisor;
        else if (src != out) memcpy((void*)(out + lo), (const void*)(src + lo), (hi - lo) * sizeof(double));
    };
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t workers = n < ((size_t)3 << 18) ? 1 : std::min<size_t>(hw ? hw : 4, 8);
    std::vector<std::thread> pool;
    for (size_t w = 1; w < workers; w++) pool.emplace_back(rows, n * w / workers, n * (w + 1) / workers);
    rows(0, n / workers);
    for (std::thread& t : pool) t.join();
    pinned_release(pin);
    return RM_OK;
}

int rm_renderer_read_sums(rm_renderer* r, rm_vec3* out) {
    if (!r || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_read_sums: null argument");
    return read_accumulator(r, out, 0.0);
}

int rm_renderer_read_frame(rm_renderer* r, size_t sample_count, rm_vec3* out) {
    if (!r || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_read_frame: null argument");
    // a zero sample_count divides by zero like the reference would (inf / NaN), it does not mean "no division"
    if (sample_count == 0) {
        if (int st = read_accumulator(r, out, 0.0)) return st;
        const size_t n = r->settings.camera_settings.backbuffer_width * r->settings.camera_settings.backbuffer_height;
        for (size_t i = 0; i < n; i++) { out[i].x /= 0.0; out[i].y /= 0.0; out[i].z /= 0.0; }
        return RM_OK;
    }
    return read_accumulator(r, out, (double)sample_count);
}

int rm_renderer_read_rgb8(rm_renderer* r, size_t sample_count, double exposure, double gamma, uint8_t* out) {
    if (!r || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_read_rgb8: null argument");
    RM_CUDA(cudaSetDevice(r->device));
    const size_t n = r->settings.camera_settings.backbuffer_width * r->settings.camera_settings.backbuffer_height;
    unsigned char* d_out = nullptr;
    RM_CUDA(dev_malloc(&d_out, n * 3));
    // sum / sample_count (src/trace.rs:95), then cli_old/src/main.rs:157-181, on the render stream: 3 B per pixel cross the bus
    int st = tonemap_device(r->accum, n, (double)sample_count, exposure, gamma, d_out, r->stream);
    if (st == RM_OK) {
        r->launches++;
        if (cudaMemcpyAsync(out, d_out, n * 3, cudaMemcpyDeviceToHost, r->stream) != cudaSuccess || cudaStreamSynchronize(r->stream) != cudaSuccess)
            st = fail(RM_ERR_CUDA, "D2H of the 8-bit image failed");
    }
    dev_free(d_out);
    harvest_events(r);
    return st;
}

int rm_renderer_read_moments(rm_renderer* r, rm_vec3* out) {
    if (!r || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_read_moments: null argument");
    if (!r->moments) return fail(RM_ERR_STATE, "rm_renderer_read_moments: the renderer was created without RM_FLAG_MOMENTS");
    return read_accumulator(r, out, 0.0, r->moments);
}

int rm_renderer_read_aovs(rm_renderer* r, size_t sample_count, rm_vec3* albedo, rm_vec3* normal, double* depth) {
    if (!r) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_read_aovs: null renderer");
    if (!r->aov) return fail(RM_ERR_STATE, "rm_renderer_read_aovs: the renderer was created without RM_FLAG_AOV");
    if (sample_count == 0) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_read_aovs: sample_count is 0");
    const size_t n = r->settings.camera_settings.backbuffer_width * r->settings.camera_settings.backbuffer_height;
    const double div = (double)sample_count;
    if (albedo) if (int st = read_accumulator(r, albedo, div, r->aov, n * 3)) return st;
    if (normal) if (int st = read_accumulator(r, normal, div, r->aov + n * 3, n * 3)) return st;
    if (depth) if (int st = read_accumulator(r, depth, div, r->aov + n * 6, n)) return st;
    return RM_OK;
}

int rm_renderer_read_denoised(rm_renderer* r, size_t sample_count, const rm_denoise_settings* settings, rm_vec3* out) {
    if (!r || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_read_denoised: null argument");
    if (!r->aov || !r->moments) return fail(RM_ERR_STATE, "rm_renderer_read_denoised: needs a renderer created with RM_FLAG_AOV and RM_FLAG_MOMENTS");
    if (r->opt.world_size > 1) return fail(RM_ERR_UNSUPPORTED, "rm_renderer_read_denoised: the filter needs the whole frame's sums (world_size > 1)");
    if (sample_count < 2) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_read_denoised: the variance needs sample_count >= 2");
    rm_denoise_settings s;
    if (int st = resolve_denoise_settings(settings, &s, "rm_renderer_read_denoised")) return st;
    RM_CUDA(cudaSetDevice(r->device));
    const size_t n = r->settings.camera_settings.backbuffer_width * r->settings.camera_settings.backbuffer_height;
    // the last pass writes the f64 frame into a pinned block; a copy moves it on to the caller's memory
    rm_vec3* pin = (rm_vec3*)pinned_acquire(std::max<size_t>(n, 1) * sizeof(rm_vec3));
    if (!pin) return fail(RM_ERR_CUDA, std::string("denoiser: ") + cudaGetErrorString(cudaErrorMemoryAllocation));
    const int st = denoise_shares_to_host(&r, 1, sample_count, s, pin);
    harvest_events(r);
    if (st == RM_OK) memcpy((void*)out, (const void*)pin, n * sizeof(rm_vec3));
    pinned_release(pin);
    return st;
}

size_t rm_renderer_tile_errors(rm_renderer* r, size_t sample_count, double* out, size_t capacity) {
    if (!r) { fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_tile_errors: null renderer"); return 0; }
    if (!r->moments) { fail(RM_ERR_STATE, "rm_renderer_tile_errors: the renderer was created without RM_FLAG_MOMENTS"); return 0; }
    if (sample_count < 2) { fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_tile_errors: the estimate needs sample_count >= 2"); return 0; }
    const rm_settings& s = r->settings;
    const size_t n_tiles = tile_layout(s.camera_settings.backbuffer_width, s.camera_settings.backbuffer_height, s.tile_size[0], s.tile_size[1]).size();
    double* pin = (double*)pinned_acquire(std::max<size_t>(n_tiles, 1) * sizeof(double));
    if (!pin) { fail(RM_ERR_OUT_OF_MEMORY, "rm_renderer_tile_errors: cannot pin the result block"); return 0; }
    for (size_t t = 0; t < n_tiles; t++) pin[t] = NAN;           // tiles of other shares stay NaN
    const Share share(r->opt);
    const int st = tile_errors_to_host(&r, 1, sample_count, pin, n_tiles, share.first_tile(), share.tile_step());
    if (st == RM_OK && out) memcpy(out, pin, std::min(n_tiles, capacity) * sizeof(double));
    pinned_release(pin);
    return st == RM_OK ? n_tiles : 0;
}

int rm_renderer_set_active_tiles(rm_renderer* r, const uint8_t* active, size_t tile_count) {
    if (!r) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_set_active_tiles: null renderer");
    const rm_settings& s = r->settings;
    const std::vector<TileRect> layout = tile_layout(s.camera_settings.backbuffer_width, s.camera_settings.backbuffer_height, s.tile_size[0], s.tile_size[1]);
    if (active && tile_count != layout.size())
        return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_set_active_tiles: tile_count is not the tile count of the layout");
    RM_CUDA(cudaSetDevice(r->device));
    // the share's pixel map holds its tiles in queue order, each as one contiguous run (build_pixel_map)
    const Share share(r->opt);
    std::vector<uint3> runs;
    size_t src = 0, n_active = 0, owned = 0;
    for (size_t t = 0; t < layout.size(); t++) {
        if (!share.owns_tile(t)) continue;
        const size_t len = layout[t].width * layout[t].height;
        if (active && active[t]) { runs.push_back(make_uint3((unsigned)src, (unsigned)n_active, (unsigned)len)); n_active += len; }
        src += len;
        owned++;
    }
    if (!active || runs.size() == owned) {          // the whole share: the shared map, as created
        r->rp.pixel_map = r->pixel_map;
        r->rp.n_pixels = (unsigned)r->pixel_map_ref->n;
        r->batch_spp = r->full_batch_spp;
        return RM_OK;
    }
    // never written to the cached shared map: the renderer gets its own compacted copy of the active runs
    if (!r->active_map) RM_CUDA(dev_malloc(&r->active_map, std::max<size_t>(r->pixel_map_ref->n, 1) * sizeof(unsigned)));
    if (!r->active_runs) RM_CUDA(dev_malloc(&r->active_runs, std::max<size_t>(owned, 1) * sizeof(uint3)));
    if (!runs.empty()) {
        RM_CUDA(cudaMemcpyAsync(r->active_runs, runs.data(), runs.size() * sizeof(uint3), cudaMemcpyHostToDevice, r->stream));
        k_gather_pixels<<<(unsigned)runs.size(), kBlock, 0, r->stream>>>(r->pixel_map, r->active_runs, r->active_map);
        r->launches++;
        RM_CUDA(cudaGetLastError());
    }
    r->rp.pixel_map = r->active_map;
    r->rp.n_pixels = (unsigned)n_active;
    // as many samples per batch as the queues hold for the active pixels (rm_renderer_render cuts a batch at the range's end)
    size_t spp = n_active ? std::max<size_t>(1, (size_t)r->rp.cap / n_active) : r->full_batch_spp;
    while (spp > 1 && spp * n_active >= 0xffffffffull) spp--;
    r->batch_spp = spp;
    return RM_OK;
}

int rm_renderer_stats(rm_renderer* r, rm_stats* out) {
    if (!r || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_stats: null argument");
    RM_CUDA(cudaSetDevice(r->device));
    RM_CUDA(cudaStreamSynchronize(r->stream));
    harvest_events(r);
    DevTotals t{};
    RM_CUDA(cudaMemcpy(&t, r->totals, sizeof(t), cudaMemcpyDeviceToHost));
    out->samples = t.samples;
    out->rays = t.rays;
    out->nonfinite_samples = t.nonfinite;
    out->kernel_launches = r->launches;
    out->device_ms = r->device_ms;
    out->upload_ms = r->ds ? r->ds->upload_ms : 0.0;
    out->upload_bytes = (r->ds ? r->ds->bytes : 0) + (uint64_t)r->uploaded_pixel_map_bytes;
    return RM_OK;
}

int rm_renderer_stage_stats(rm_renderer* r, rm_stage_stats* out) {
    if (!r || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_renderer_stage_stats: null argument");
    RM_CUDA(cudaSetDevice(r->device));
    RM_CUDA(cudaStreamSynchronize(r->stream));
    harvest_events(r);
    DevTotals t{};
    RM_CUDA(cudaMemcpy(&t, r->totals, sizeof(t), cudaMemcpyDeviceToHost));
    for (int i = 0; i < RM_STAGE_SLOTS; i++) {
        for (int k = 0; k < RM_KERNEL_KINDS; k++) { out->ms[k][i] = r->stage_ms[k][i]; out->launches[k][i] = r->stage_launches[k][i]; }
        out->rays[i] = t.stage_rays[i];
        out->grid_rays[i] = t.grid_rays[i];
        out->cells[i] = t.cells[i];
        out->triangle_tests[i] = t.tests[i];
        out->shaded_triangles[i] = t.shaded[i];
        out->evaluated_tests[i] = t.survivors[i];
        out->occupied_cells[i] = t.occupied[i];
        out->evaluated_test_flops[i] = t.test_flops[i];
        out->cell_sphere_tests[i] = t.cell_tests[i];
    }
    return RM_OK;
}

void rm_renderer_destroy(rm_renderer* r) { delete r; }

// 8 independent chains per thread of alternating DMUL / DADD (this file is compiled with -fmad=false: they stay two instructions)
__global__ void __launch_bounds__(256) k_fp64_rate(double* out, int iters, double m, double c) {
    double a[8];
#pragma unroll
    for (int j = 0; j < 8; j++) a[j] = 1.0 + 1e-3 * (double)(threadIdx.x + j);
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) { a[j] = a[j] * m; a[j] = a[j] + c; }
    }
    double sum = 0.0;
#pragma unroll
    for (int j = 0; j < 8; j++) sum += a[j];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = sum;
}

int rm_measure_fp64_rate(int device, double* gops_out) {
    if (!gops_out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_measure_fp64_rate: null argument");
    RM_CUDA(cudaSetDevice(device));
    const int sms = sm_count(device), blocks = sms * 8, iters = 4096;
    double* out = nullptr;
    RM_CUDA(dev_malloc(&out, (size_t)blocks * 256 * sizeof(double)));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 0.f;
    cudaError_t e = cudaSuccess;
    for (int rep = 0; rep < 4 && e == cudaSuccess; rep++) {          // rep 0 warms up
        cudaEventRecord(e0, 0);
        k_fp64_rate<<<blocks, 256>>>(out, iters, 0.9999999, 1e-7);
        cudaEventRecord(e1, 0);
        e = cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && (best == 0.f || ms < best)) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    dev_free(out);
    if (e != cudaSuccess || best <= 0.f) return fail(RM_ERR_CUDA, std::string("fp64 rate kernel: ") + cudaGetErrorString(e));
    *gops_out = (double)blocks * 256.0 * (double)iters * 16.0 / ((double)best * 1e-3) / 1e9;
    return RM_OK;
}

/* Hand the cached device memory (stream-ordered pool of every visible device) and the cached pinned staging blocks back. */
int rm_release_cached_memory(void) {
    {
        std::lock_guard<std::mutex> lk(g_pixel_map_mu);
        pixel_map_cache_trim(0);
    }
    int count = 0;
    int before = 0;
    cudaGetDevice(&before);
    visible_cache_clear();
    cudaSetDevice(before);
    if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); count = 0; }
    int current = 0;
    if (count) cudaGetDevice(&current);
    for (int d = 0; d < count; d++) {
        cudaMemPool_t pool = nullptr;
        {
            std::lock_guard<std::mutex> lk(g_pool_mu);
            auto it = g_pools.find(d);
            if (it != g_pools.end()) pool = it->second;
        }
        if (pool && cudaSetDevice(d) == cudaSuccess && cudaDeviceSynchronize() == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
        cudaGetLastError();
    }
    if (count) cudaSetDevice(current);
    {
        std::lock_guard<std::mutex> lk(g_pin_mu);
        for (PinnedBlock& f : g_pin_free) cudaFreeHost(f.p);
        g_pin_free.clear();
    }
    return RM_OK;
}

#if defined(RM_TRAV_PROFILE)
// profiling builds only: cycles per k_traverse phase {refill, walk, tests, finish, loop head, -, -, warps}; reading resets
int rm_debug_trav_profile(unsigned long long* out8) {
    cudaDeviceSynchronize();
    unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    cudaMemcpyFromSymbol(out8, g_trav_prof, sizeof(z));
    cudaMemcpyToSymbol(g_trav_prof, z, sizeof(z));
    return RM_OK;
}
#endif

}  // extern "C"
