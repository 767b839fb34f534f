// rm_host.cpp — host side of the C ABI: meshes, the uniform grid, scenes, tile layout.
// Setup-path code (runs once per scene); everything per ray / per sample is CUDA (rm_device.cu).
// Citations are relative to the reference checkout (Nyrox/raymond).

#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <limits>
#include <thread>

#include "rm_internal.hpp"

namespace rm {

static thread_local std::string g_last_error;
static thread_local int g_last_status = RM_OK;

void set_error(const std::string& msg) { g_last_error = msg; if (g_last_status == RM_OK) g_last_status = RM_ERR_INVALID_ARGUMENT; }
int fail(int status, const std::string& msg) { g_last_error = msg; g_last_status = status; return status; }

// generate_primary_ray_with_dof (src/trace.rs:335-360) rejection-samples the aperture disk until a point lies strictly inside
// it, then unwraps the focal-plane hit.  An infinite radius, one whose square overflows (dx² + dy² = ∞) or a non-finite
// position makes every distance ∞ or NaN, so the loop never ends; a negative or NaN focal length makes the unwrap panic.
int validate_camera(const rm_camera_settings& c, const char* who) {
    if (!(c.aperture_radius > 0.0)) return RM_OK;   // the pinhole camera (D2)
    if (!(c.aperture_radius <= 1e150))
        return fail(RM_ERR_INVALID_ARGUMENT, std::string(who) + ": aperture_radius must be <= 1e150 (a larger one never finishes the aperture sampling)");
    if (!std::isfinite(c.position.x) || !std::isfinite(c.position.y) || !std::isfinite(c.position.z))
        return fail(RM_ERR_INVALID_ARGUMENT, std::string(who) + ": a depth-of-field camera needs a finite position");
    if (!(c.focal_length >= 0.0))
        return fail(RM_ERR_INVALID_ARGUMENT, std::string(who) + ": a depth-of-field camera needs focal_length >= 0 (the focal plane must be in front of it)");
    return RM_OK;
}

// ------------------------------------------------------------------ bounds

// The reference seeds its min/max folds with these odd sentinels (mesh.rs:124-125,
// triangle.rs:71-72); a mesh outside that box gets "wrong" bounds there, and so here.
static const double kMinSeed[3] = {125125.0, 1251251.0, 12512512.0};
static const double kMaxSeed[3] = {-123125.0, -125123.0, -512123.0};

static inline const double* pos(const rm_vertex& v) { return &v.position.x; }

static inline void fold_triangle(const rm_triangle& t, double mn[3], double mx[3]) {
    const double* p[3] = {pos(t.v0), pos(t.v1), pos(t.v2)};
    for (int a = 0; a < 3; a++)
        for (int k = 0; k < 3; k++) {
            mn[a] = std::fmin(mn[a], p[k][a]);   // f64::min ignores NaN, like fmin
            mx[a] = std::fmax(mx[a], p[k][a]);
        }
}

rm_aabb mesh_bounds(const rm_triangle* tris, size_t n) {
    double mn[3] = {kMinSeed[0], kMinSeed[1], kMinSeed[2]};
    double mx[3] = {kMaxSeed[0], kMaxSeed[1], kMaxSeed[2]};
    for (size_t i = 0; i < n; i++) fold_triangle(tris[i], mn, mx);
    return rm_aabb{{mn[0], mn[1], mn[2]}, {mx[0], mx[1], mx[2]}};
}

// ------------------------------------------------------------------ grid build

// Rust `x as usize` (saturating, NaN -> 0)                 acc_grid.rs:13-15
static inline uint64_t saturating_usize(double v) {
    if (!(v > 0.0)) return 0;
    if (v >= 18446744073709551616.0) return std::numeric_limits<uint64_t>::max();
    return (uint64_t)v;
}

// cgmath `cast::<usize>()`: Some(trunc toward zero) iff -1 < v < 2^64   acc_grid.rs:46,50
static inline bool checked_usize(double v, uint64_t* out) {
    if (!(v > -1.0 && v < 18446744073709551616.0)) return false;
    *out = (uint64_t)v;
    return true;
}

struct CellRange { uint64_t lo[3], hi[3]; };

// estimate_grid_resolution + cell_size                      acc_grid.rs:6-17,38 — shared by the host and the device build
int grid_dims(const rm_aabb& bounds, size_t n, uint64_t res[3], double cell[3]) {
    const double size[3] = {bounds.max.x - bounds.min.x, bounds.max.y - bounds.min.y, bounds.max.z - bounds.min.z};
    const double volume = std::fabs(size[0] * size[1] * size[2]);
    const double density = std::pow((3.0 * (double)n) / volume, 1.0 / 3.0);
    for (int a = 0; a < 3; a++) res[a] = saturating_usize(std::fabs(size[a]) * density);
    if (res[0] == 0 || res[1] == 0 || res[2] == 0)
        return fail(RM_ERR_DEGENERATE_BOUNDS, "grid resolution has a zero axis (reference: `grid_res[i] - 1` underflows, acc_grid.rs:54)");
    for (int a = 0; a < 3; a++) cell[a] = size[a] / (double)res[a];
    if (res[0] > 0x7fffffffull || res[1] > 0x7fffffffull || res[2] > 0x7fffffffull)
        return fail(RM_ERR_UNSUPPORTED, "grid resolution exceeds 2^31 - 1 on an axis");
    const long double cells_ld = (long double)res[0] * (long double)res[1] * (long double)res[2];
    if (cells_ld >= 4294967295.0L) return fail(RM_ERR_UNSUPPORTED, "grid has 2^32 or more cells");
    if (n >= 0xffffffffull) return fail(RM_ERR_UNSUPPORTED, "mesh has 2^32 or more triangles");
    return RM_OK;
}

int build_grid(std::vector<rm_triangle>&& tris, const rm_aabb& bounds, std::shared_ptr<Grid>* out) {
    auto g = std::make_shared<Grid>();
    const size_t n = tris.size();
    const double bmin[3] = {bounds.min.x, bounds.min.y, bounds.min.z};
    uint64_t res[3];
    double cell[3];
    if (int st = grid_dims(bounds, n, res, cell)) return st;
    const uint64_t n_cells = res[0] * res[1] * res[2];

    // pass 1: per-triangle cell range (acc_grid.rs:43-56), per-cell counts
    std::vector<CellRange> ranges(n);
    std::vector<uint32_t>& start = g->cell_start;
    start.assign(n_cells + 1, 0);
    uint64_t total = 0;
    for (size_t i = 0; i < n; i++) {
        double mn[3] = {kMinSeed[0], kMinSeed[1], kMinSeed[2]};
        double mx[3] = {kMaxSeed[0], kMaxSeed[1], kMaxSeed[2]};
        fold_triangle(tris[i], mn, mx);                     // Triangle::find_bounds  triangle.rs:70-84
        CellRange& r = ranges[i];
        for (int a = 0; a < 3; a++) {
            if (!checked_usize((mn[a] - bmin[a]) / cell[a], &r.lo[a]) || !checked_usize((mx[a] - bmin[a]) / cell[a], &r.hi[a]))
                return fail(RM_ERR_GRID_CAST, "Failed to cast cell bounds to usize (acc_grid.rs:47,51)");
            r.lo[a] = std::min(r.lo[a], res[a] - 1);
            r.hi[a] = std::min(r.hi[a], res[a] - 1);
        }
        for (uint64_t z = r.lo[2]; z <= r.hi[2]; z++)
            for (uint64_t y = r.lo[1]; y <= r.hi[1]; y++) {
                // the reference strides z by res.z, not res.y (acc_grid.rs:61) — kept
                const uint64_t row = res[0] * (y + z * res[2]);
                if (row + r.hi[0] >= n_cells)
                    return fail(RM_ERR_GRID_INDEX_OOB, "cell index out of bounds while inserting triangle " + std::to_string(i) +
                                                           " (reference panics at acc_grid.rs:61)");
                for (uint64_t x = r.lo[0]; x <= r.hi[0]; x++) start[row + x + 1]++;
                total += r.hi[0] - r.lo[0] + 1;
            }
    }
    if (total >= 0xffffffffull) return fail(RM_ERR_UNSUPPORTED, "grid has 2^32 or more triangle references");
    // exclusive scan
    for (uint64_t c = 0; c < n_cells; c++) start[c + 1] += start[c];
    // pass 2: fill in ascending triangle order (the reference pushes indices in mesh order)
    g->references.resize(total);
    std::vector<uint32_t> cursor(start.begin(), start.end() - 1);
    for (size_t i = 0; i < n; i++) {
        const CellRange& r = ranges[i];
        for (uint64_t z = r.lo[2]; z <= r.hi[2]; z++)
            for (uint64_t y = r.lo[1]; y <= r.hi[1]; y++) {
                const uint64_t row = res[0] * (y + z * res[2]);
                for (uint64_t x = r.lo[0]; x <= r.hi[0]; x++) g->references[cursor[row + x]++] = (uint32_t)i;
            }
    }
    g->triangles = std::move(tris);
    g->bounds = bounds;
    for (int a = 0; a < 3; a++) g->resolution[a] = res[a];
    g->cell_size = rm_vec3{cell[0], cell[1], cell[2]};
    *out = g;
    return RM_OK;
}

// ------------------------------------------------------------------ tiles

std::vector<TileRect> tile_layout(size_t W, size_t H, size_t tw, size_t th) {
    // column-major: y advances first, edge tiles clipped   src/trace.rs:146-172
    std::vector<TileRect> out;
    if (W == 0 || H == 0 || tw == 0 || th == 0) return out;
    for (size_t x = 0; x < W; x += tw)
        for (size_t y = 0; y < H; y += th) out.push_back(TileRect{x, y, std::min(tw, W - x), std::min(th, H - y)});
    return out;
}

// ------------------------------------------------------------------ PLY

// Mesh::load_ply                                          mesh.rs:58-121
// ASCII only; the header is only scanned for `element vertex N`; a vertex line needs >= 6 numbers
// (x y z nx ny nz [s t]); face lines are read to EOF and anything but a triangle is dropped.
namespace {

struct LineReader {
    const char* p;
    const char* end;
    bool next(const char** b, const char** e) {
        if (p >= end) return false;
        const char* nl = (const char*)memchr(p, '\n', (size_t)(end - p));
        const char* stop = nl ? nl : end;
        *b = p;
        *e = (stop > p && stop[-1] == '\r') ? stop - 1 : stop;
        p = nl ? nl + 1 : end;
        return true;
    }
};

inline void skip_ws(const char*& b, const char* e) { while (b < e && (*b == ' ' || *b == '\t' || *b == '\v' || *b == '\f' || *b == '\r')) b++; }
inline bool token(const char*& b, const char* e, const char** tb, const char** te) {
    skip_ws(b, e);
    if (b >= e) return false;
    *tb = b;
    while (b < e && !(*b == ' ' || *b == '\t' || *b == '\v' || *b == '\f' || *b == '\r')) b++;
    *te = b;
    return true;
}
inline bool tok_eq(const char* tb, const char* te, const char* s) { size_t n = strlen(s); return (size_t)(te - tb) == n && memcmp(tb, s, n) == 0; }

inline bool parse_f64(const char* tb, const char* te, double* out) {
    if (tb < te && *tb == '+') tb++;                       // Rust's f64::from_str accepts a leading '+'
    auto r = std::from_chars(tb, te, *out);
    return r.ec == std::errc() && r.ptr == te;
}
inline bool parse_u32(const char* tb, const char* te, uint32_t* out) {
    if (tb < te && *tb == '+') tb++;
    auto r = std::from_chars(tb, te, *out);
    return r.ec == std::errc() && r.ptr == te;
}

// Vertex::calculate_tangent                               vertex.rs:13-27
rm_vec3 face_tangent(const rm_vertex& x, const rm_vertex& y, const rm_vertex& z) {
    const double e1[3] = {y.position.x - x.position.x, y.position.y - x.position.y, y.position.z - x.position.z};
    const double e2[3] = {z.position.x - x.position.x, z.position.y - x.position.y, z.position.z - x.position.z};
    const double u1x = y.uv.x - x.uv.x, u1y = y.uv.y - x.uv.y;
    const double u2x = z.uv.x - x.uv.x, u2y = z.uv.y - x.uv.y;
    const double f = 1.0 / (u1x * u2y - u2x * u1y);
    double t[3];
    for (int a = 0; a < 3; a++) t[a] = f * (u2y * e1[a] - u1y * e2[a]);
    const double inv = 1.0 / std::sqrt((t[0] * t[0] + t[1] * t[1]) + t[2] * t[2]);
    return rm_vec3{t[0] * inv, t[1] * inv, t[2] * inv};
}

}  // namespace

int load_ply(const char* path, Mesh* mesh);
int load_ply(const char* path, Mesh* mesh) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    if (!f) return fail(RM_ERR_IO, std::string("cannot read ") + path);
    std::streamsize len = f.tellg();
    f.seekg(0);
    std::string buf((size_t)len, '\0');
    if (len > 0 && !f.read(&buf[0], len)) return fail(RM_ERR_IO, std::string("cannot read ") + path);

    LineReader lr{buf.data(), buf.data() + buf.size()};
    const char *b, *e, *tb, *te;
    size_t n_vertices = 0;
    bool header_done = false;
    while (lr.next(&b, &e)) {
        if (!token(b, e, &tb, &te)) return fail(RM_ERR_PLY, "empty line inside the PLY header (mesh.rs:69 unwrap)");
        if (tok_eq(tb, te, "element")) {
            if (!token(b, e, &tb, &te)) return fail(RM_ERR_PLY, "`element` without a name");
            if (tok_eq(tb, te, "vertex")) {
                uint64_t nv = 0;
                if (!token(b, e, &tb, &te)) return fail(RM_ERR_PLY, "`element vertex` without a count");
                auto r = std::from_chars(tb, te, nv);
                if (r.ec != std::errc() || r.ptr != te) return fail(RM_ERR_PLY, "bad vertex count");
                n_vertices = (size_t)nv;
            }
        } else if (tok_eq(tb, te, "end_header")) {
            header_done = true;
            break;
        }
    }
    (void)header_done;   // a header without end_header just leaves no lines for the vertex loop

    // The body is parsed by a few host threads: line starts are collected in one pass, vertex lines and face lines are
    // independent of each other (a face's tangent is computed from the three vertices' positions and uvs and stored in
    // ITS copies of them, mesh.rs:101-114).  The first failure in line order is the one reported, as a sequential reader would.
    std::vector<std::pair<const char*, const char*>> lines;
    lines.reserve((size_t)(lr.end - lr.p) / 24 + 16);
    while (lr.next(&b, &e)) lines.emplace_back(b, e);
    const size_t n_vlines = std::min(n_vertices, lines.size());
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t workers = lines.size() < 20000 ? 1 : std::min<size_t>(hw ? hw : 4, 16);
    struct Failure { size_t line = (size_t)-1; std::string msg; };
    auto first_failure = [](const std::vector<Failure>& f) { size_t best = 0; for (size_t i = 1; i < f.size(); i++) if (f[i].line < f[best].line) best = i; return f[best]; };

    std::unique_ptr<rm_vertex[]> vertices(new rm_vertex[std::max<size_t>(n_vlines, 1)]);   // first touched by the parsing threads
    {
        std::vector<Failure> fails(workers);
        auto parse_vertices = [&](size_t w) {
            const char *tb, *te;
            for (size_t i = n_vlines * w / workers; i < n_vlines * (w + 1) / workers; i++) {
                const char* b = lines[i].first;
                const char* e = lines[i].second;
                double v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                int k = 0;
                while (token(b, e, &tb, &te)) {
                    double x;
                    if (!parse_f64(tb, te, &x)) { fails[w] = Failure{i, "vertex line " + std::to_string(i) + " holds a non-number (mesh.rs:83 unwrap)"}; return; }
                    if (k < 8) v[k] = x;
                    k++;
                }
                if (k < 6) { fails[w] = Failure{i, "vertex line " + std::to_string(i) + " has fewer than 6 numbers (mesh.rs:85-86 index)"}; return; }
                rm_vertex& vx = vertices[i];
                vx.position = rm_vec3{v[0], v[1], v[2]};
                vx.normal = rm_vec3{v[3], v[4], v[5]};
                vx.uv = rm_vec2{k > 6 ? v[6] : 0.0, k > 7 ? v[7] : 0.0};
                vx.tangent = rm_vec3{0.0, 0.0, 0.0};
            }
        };
        std::vector<std::thread> pool;
        for (size_t w = 1; w < workers; w++) pool.emplace_back(parse_vertices, w);
        parse_vertices(0);
        for (std::thread& t : pool) t.join();
        const Failure f = first_failure(fails);
        if (f.line != (size_t)-1) return fail(RM_ERR_PLY, f.msg);
        if (lines.size() < n_vertices) return fail(RM_ERR_PLY, "PLY ends inside the vertex list (mesh.rs:81 unwrap)");
    }

    std::vector<rm_triangle> faces;
    {
        const size_t n_flines = lines.size() - n_vlines;
        std::vector<Failure> fails(workers);
        struct Tri { uint32_t a, b, c; };
        std::vector<std::vector<Tri>> part(workers);
        auto parse_faces = [&](size_t w) {
            const char *tb, *te;
            std::vector<Tri>& out = part[w];
            const size_t lo = n_flines * w / workers, hi = n_flines * (w + 1) / workers;
            out.reserve(hi - lo);
            for (size_t i = lo; i < hi; i++) {
                const char* b = lines[n_vlines + i].first;
                const char* e = lines[n_vlines + i].second;
                uint32_t idx[4];
                int k = 0;
                while (token(b, e, &tb, &te)) {
                    uint32_t x;
                    if (!parse_u32(tb, te, &x)) { fails[w] = Failure{i, "face line holds a non-u32 token (mesh.rs:95 unwrap)"}; return; }
                    if (k < 4) idx[k] = x;
                    k++;
                }
                if (k == 0) { fails[w] = Failure{i, "empty line in the face list (mesh.rs:97 index)"}; return; }
                if (idx[0] != 3) continue;                          // non-triangles are silently dropped (mesh.rs:116)
                if (k < 4) { fails[w] = Failure{i, "triangle face with fewer than 3 indices"}; return; }
                for (int j = 1; j <= 3; j++)
                    if (idx[j] >= n_vlines) { fails[w] = Failure{i, "face index out of range (mesh.rs:102-104 index)"}; return; }
                out.push_back(Tri{idx[1], idx[2], idx[3]});
            }
        };
        {
            std::vector<std::thread> pool;
            for (size_t w = 1; w < workers; w++) pool.emplace_back(parse_faces, w);
            parse_faces(0);
            for (std::thread& t : pool) t.join();
        }
        const Failure f = first_failure(fails);
        if (f.line != (size_t)-1) return fail(RM_ERR_PLY, f.msg);
        std::vector<size_t> offset(workers + 1, 0);
        for (size_t w = 0; w < workers; w++) offset[w + 1] = offset[w] + part[w].size();
        faces.resize(offset[workers]);
        auto build = [&](size_t w) {
            for (size_t i = 0; i < part[w].size(); i++) {
                const Tri& x = part[w][i];
                rm_triangle& t = faces[offset[w] + i];
                t = rm_triangle{vertices[x.a], vertices[x.b], vertices[x.c]};
                const rm_vec3 tg = face_tangent(t.v0, t.v1, t.v2);       // the face's tangent goes into its copies of the vertices
                t.v0.tangent = tg; t.v1.tangent = tg; t.v2.tangent = tg;
            }
        };
        std::vector<std::thread> pool;
        for (size_t w = 1; w < workers; w++) pool.emplace_back(build, w);
        build(0);
        for (std::thread& t : pool) t.join();
    }
    mesh->triangles = std::move(faces);
    mesh->bounds = mesh_bounds(mesh->triangles.data(), mesh->triangles.size());
    return RM_OK;
}

}  // namespace rm

// ==================================================================== C ABI

using namespace rm;

extern "C" {

const char* rm_last_error(void) { return g_last_error.c_str(); }
int rm_last_status(void) { return g_last_status; }
int rm_abi_version(void) { return RM_ABI_VERSION; }

rm_mesh* rm_mesh_from_triangles(const rm_triangle* triangles, size_t count) {
    if (!triangles && count) { set_error("rm_mesh_from_triangles: null triangles"); return nullptr; }
    rm_mesh* m = new (std::nothrow) rm_mesh();
    if (!m) { set_error("out of memory"); return nullptr; }
    try {
        m->mesh.triangles.assign(triangles, triangles + count);
    } catch (const std::bad_alloc&) {
        delete m; set_error("out of memory"); return nullptr;
    }
    m->mesh.bounds = mesh_bounds(m->mesh.triangles.data(), count);
    return m;
}

rm_mesh* rm_mesh_load_ply(const char* path) {
    if (!path) { set_error("rm_mesh_load_ply: null path"); return nullptr; }
    rm_mesh* m = new (std::nothrow) rm_mesh();
    if (!m) { set_error("out of memory"); return nullptr; }
    try {
        if (load_ply(path, &m->mesh) != RM_OK) { delete m; return nullptr; }
    } catch (const std::bad_alloc&) {
        delete m; set_error("out of memory"); return nullptr;
    }
    return m;
}

int rm_mesh_translate(rm_mesh* mesh, rm_vec3 t) {
    if (!mesh) return fail(RM_ERR_INVALID_ARGUMENT, "rm_mesh_translate: null mesh");
    for (rm_triangle& tri : mesh->mesh.triangles) {
        rm_vertex* v[3] = {&tri.v0, &tri.v1, &tri.v2};
        for (int k = 0; k < 3; k++) { v[k]->position.x += t.x; v[k]->position.y += t.y; v[k]->position.z += t.z; }
    }
    mesh->mesh.bounds = mesh_bounds(mesh->mesh.triangles.data(), mesh->mesh.triangles.size());
    return RM_OK;
}

size_t rm_mesh_triangle_count(const rm_mesh* mesh) { return mesh ? mesh->mesh.triangles.size() : 0; }

int rm_mesh_bounds(const rm_mesh* mesh, rm_aabb* out) {
    if (!mesh || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_mesh_bounds: null argument");
    *out = mesh->mesh.bounds;
    return RM_OK;
}

int rm_mesh_triangles(const rm_mesh* mesh, size_t first, size_t count, rm_triangle* out) {
    if (!mesh || (!out && count)) return fail(RM_ERR_INVALID_ARGUMENT, "rm_mesh_triangles: null argument");
    if (first > mesh->mesh.triangles.size() || count > mesh->mesh.triangles.size() - first)
        return fail(RM_ERR_INVALID_ARGUMENT, "rm_mesh_triangles: range out of bounds");
    if (count) memcpy(out, mesh->mesh.triangles.data() + first, count * sizeof(rm_triangle));
    return RM_OK;
}

void rm_mesh_destroy(rm_mesh* mesh) { delete mesh; }

rm_grid* rm_grid_build(rm_mesh* mesh, int* status) {
    int st = RM_OK;
    rm_grid* out = nullptr;
    if (!mesh) {
        st = fail(RM_ERR_INVALID_ARGUMENT, "rm_grid_build: null mesh");
    } else {
        try {
            std::shared_ptr<Grid> g;
            rm_aabb bounds = mesh->mesh.bounds;
            std::vector<rm_triangle> tris = std::move(mesh->mesh.triangles);   // the Rust call moves the Mesh
            mesh->mesh.triangles.clear();
            mesh->mesh.bounds = mesh_bounds(nullptr, 0);
            st = build_grid(std::move(tris), bounds, &g);
            if (st == RM_OK) { out = new rm_grid(); out->grid = g; }
        } catch (const std::bad_alloc&) {
            st = fail(RM_ERR_OUT_OF_MEMORY, "out of memory while building the grid");
        }
    }
    if (status) *status = st;
    return out;
}

rm_grid* rm_grid_build_on_device(rm_mesh* mesh, int device, int* status) {
    int st = RM_OK;
    rm_grid* out = nullptr;
    if (!mesh) {
        st = fail(RM_ERR_INVALID_ARGUMENT, "rm_grid_build_on_device: null mesh");
    } else {
        try {
            std::shared_ptr<Grid> g;
            rm_aabb bounds = mesh->mesh.bounds;
            std::vector<rm_triangle> tris = std::move(mesh->mesh.triangles);   // the Rust call moves the Mesh
            mesh->mesh.triangles.clear();
            mesh->mesh.bounds = mesh_bounds(nullptr, 0);
            st = build_grid_device(std::move(tris), bounds, device, &g);
            if (st == RM_OK) { out = new rm_grid(); out->grid = g; }
        } catch (const std::bad_alloc&) {
            st = fail(RM_ERR_OUT_OF_MEMORY, "out of memory while building the grid");
        }
    }
    if (status) *status = st;
    return out;
}

rm_grid* rm_grid_retain(rm_grid* grid) { if (grid) grid->refs.fetch_add(1); return grid; }
void rm_grid_release(rm_grid* grid) { if (grid && grid->refs.fetch_sub(1) == 1) delete grid; }

int rm_grid_get_info(const rm_grid* grid, rm_grid_info* out) {
    if (!grid || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_grid_get_info: null argument");
    const Grid& g = *grid->grid;
    for (int a = 0; a < 3; a++) out->resolution[a] = (size_t)g.resolution[a];
    out->cell_size = g.cell_size;
    out->bounds = g.bounds;
    out->cell_count = (size_t)g.n_cells();
    out->reference_count = g.references.size();
    out->triangle_count = g.triangles.size();
    return RM_OK;
}

int rm_grid_get_cells(const rm_grid* grid, uint32_t* cell_start, uint32_t* references) {
    if (!grid) return fail(RM_ERR_INVALID_ARGUMENT, "rm_grid_get_cells: null grid");
    const Grid& g = *grid->grid;
    if (cell_start) memcpy(cell_start, g.cell_start.data(), g.cell_start.size() * sizeof(uint32_t));
    if (references && !g.references.empty()) memcpy(references, g.references.data(), g.references.size() * sizeof(uint32_t));
    return RM_OK;
}

rm_scene* rm_scene_create(void) { return new (std::nothrow) rm_scene(); }

static int check_material(const rm_material* m) {
    if (!m) return fail(RM_ERR_INVALID_ARGUMENT, "null material");
    if (m->kind > RM_MATERIAL_EMISSION) return fail(RM_ERR_INVALID_ARGUMENT, "unknown material kind");
    return RM_OK;
}

int rm_scene_add_sphere(rm_scene* scene, rm_vec3 origin, double radius, const rm_material* material) {
    if (!scene) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_add_sphere: null scene");
    if (int st = check_material(material)) return st;
    Object o{};
    o.geometry = GEOM_SPHERE; o.origin = origin; o.normal = rm_vec3{0, 0, 0}; o.radius = radius; o.material = *material;
    scene->objects.push_back(o);
    return RM_OK;
}

int rm_scene_add_plane(rm_scene* scene, rm_vec3 origin, rm_vec3 normal, const rm_material* material) {
    if (!scene) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_add_plane: null scene");
    if (int st = check_material(material)) return st;
    Object o{};
    o.geometry = GEOM_PLANE; o.origin = origin; o.normal = normal; o.radius = 0.0; o.material = *material;
    scene->objects.push_back(o);
    return RM_OK;
}

int rm_scene_add_grid(rm_scene* scene, rm_grid* grid, const rm_material* material) {
    if (!scene || !grid) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_add_grid: null argument");
    if (int st = check_material(material)) return st;
    Object o{};
    o.geometry = GEOM_GRID; o.origin = rm_vec3{0, 0, 0}; o.normal = rm_vec3{0, 0, 0}; o.radius = 0.0; o.grid = grid->grid; o.material = *material;
    scene->objects.push_back(o);
    return RM_OK;
}

size_t rm_scene_object_count(const rm_scene* scene) { return scene ? scene->objects.size() : 0; }
void rm_scene_destroy(rm_scene* scene) { delete scene; }

int rm_scene_set_environment(rm_scene* scene, const rm_environment* env) {
    if (!scene) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_environment: null scene");
    if (!env) { scene->env.reset(); return RM_OK; }
    if (!env->texels) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_environment: null texels");
    if (env->width < 1 || env->width > 32768 || env->height < 1 || env->height > 32768)
        return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_environment: width and height must be 1..32768");
    if (!std::isfinite(env->scale) || env->scale < 0.0) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_environment: scale must be finite and >= 0");
    if (!std::isfinite(env->rotation)) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_environment: rotation must be finite");
    const size_t n = env->width * env->height;
    for (size_t i = 0; i < 3 * n; i++)
        if (!std::isfinite(env->texels[i]) || env->texels[i] < 0.0f)
            return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_environment: texel value " + std::to_string(i) + " is negative, NaN or infinite");
    auto e = std::make_shared<Environment>();
    try {
        e->rgba.resize(4 * n);
    } catch (const std::bad_alloc&) {
        return fail(RM_ERR_OUT_OF_MEMORY, "rm_scene_set_environment: cannot hold the texels");
    }
    for (size_t i = 0; i < n; i++) {
        e->rgba[4 * i] = env->texels[3 * i];
        e->rgba[4 * i + 1] = env->texels[3 * i + 1];
        e->rgba[4 * i + 2] = env->texels[3 * i + 2];
        e->rgba[4 * i + 3] = 0.0f;
    }
    e->width = env->width;
    e->height = env->height;
    e->scale = env->scale;
    e->rotation = env->rotation;
    scene->env = std::move(e);       // placements made before keep the map they share
    return RM_OK;
}

int rm_scene_set_texture(rm_scene* scene, size_t object_index, const rm_texture* texture) {
    if (!scene) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_texture: null scene");
    if (object_index >= scene->objects.size())
        return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_texture: object index " + std::to_string(object_index) + " out of range");
    Object& o = scene->objects[object_index];
    if (!texture) { o.texture.reset(); return RM_OK; }
    if (o.material.kind == RM_MATERIAL_EMISSION) return fail(RM_ERR_UNSUPPORTED, "rm_scene_set_texture: an Emission object cannot be textured");
    if (!texture->texels) return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_texture: null texels");
    if (texture->width < 1 || texture->width > 32768 || texture->height < 1 || texture->height > 32768)
        return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_texture: width and height must be 1..32768");
    if (!std::isfinite(texture->scale_u) || !std::isfinite(texture->scale_v))
        return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_texture: scale_u and scale_v must be finite");
    const size_t n = texture->width * texture->height;
    for (size_t i = 0; i < 3 * n; i++)
        if (!std::isfinite(texture->texels[i]) || texture->texels[i] < 0.0f)
            return fail(RM_ERR_INVALID_ARGUMENT, "rm_scene_set_texture: texel value " + std::to_string(i) + " is negative, NaN or infinite");
    auto t = std::make_shared<Texture>();
    try {
        t->rgba.resize(4 * n);
    } catch (const std::bad_alloc&) {
        return fail(RM_ERR_OUT_OF_MEMORY, "rm_scene_set_texture: cannot hold the texels");
    }
    for (size_t i = 0; i < n; i++) {
        t->rgba[4 * i] = texture->texels[3 * i];
        t->rgba[4 * i + 1] = texture->texels[3 * i + 1];
        t->rgba[4 * i + 2] = texture->texels[3 * i + 2];
        t->rgba[4 * i + 3] = 0.0f;
    }
    t->width = texture->width;
    t->height = texture->height;
    t->scale_u = texture->scale_u;
    t->scale_v = texture->scale_v;
    o.texture = std::move(t);        // placements made before keep the texture they share
    return RM_OK;
}

// Radiance RGBE (.hdr) body: see rm_load_hdr in include/raymond.h.  `texels` NULL = size only.
static int decode_hdr(const std::string& buf, const char* path, size_t* width, size_t* height, float* texels) {
    auto bad = [&](const std::string& why) { return fail(RM_ERR_IMAGE, std::string(path) + ": " + why); };
    size_t p = 0;
    auto line = [&](std::string* out) {
        const size_t e = buf.find('\n', p);
        if (e == std::string::npos) return false;
        *out = buf.substr(p, e - p);
        p = e + 1;
        return true;
    };
    std::string l;
    if (!line(&l) || (l != "#?RADIANCE" && l != "#?RGBE")) return bad("not a Radiance RGBE file (no #?RADIANCE / #?RGBE line)");
    for (;;) {
        if (!line(&l)) return bad("header does not end");
        if (l.empty()) break;
        if (l.compare(0, 7, "FORMAT=") == 0 && l != "FORMAT=32-bit_rle_rgbe") return bad("unsupported " + l);
    }
    if (!line(&l)) return bad("no resolution line");
    char ys[3] = {0}, xs[3] = {0};
    unsigned long long H = 0, W = 0;
    int used = 0;
    if (sscanf(l.c_str(), "%2s %llu %2s %llu%n", ys, &H, xs, &W, &used) != 4 || (size_t)used != l.size())
        return bad("malformed resolution line");
    if (strcmp(ys, "-Y") != 0 || strcmp(xs, "+X") != 0) return bad("unsupported orientation \"" + l + "\" (only -Y H +X W)");
    if (W < 1 || H < 1 || W > ((size_t)1 << 31) / H) return bad("unsupported size " + std::to_string(W) + " x " + std::to_string(H));
    *width = (size_t)W;
    *height = (size_t)H;
    if (!texels) return RM_OK;
    const unsigned char* b = (const unsigned char*)buf.data();
    const size_t n = buf.size();
    std::vector<unsigned char> row((size_t)W * 4);
    for (size_t y = 0; y < H; y++) {
        const bool rle = W >= 8 && W <= 32767 && p + 4 <= n && b[p] == 2 && b[p + 1] == 2 && !(b[p + 2] & 0x80);
        if (rle) {
            if ((((size_t)b[p + 2] << 8) | b[p + 3]) != W) return bad("scanline " + std::to_string(y) + ": run-length width differs");
            p += 4;
            for (int c = 0; c < 4; c++)
                for (size_t x = 0; x < W;) {
                    if (p >= n) return bad("truncated");
                    size_t count = b[p++];
                    if (count > 128) {
                        count -= 128;
                        if (p >= n) return bad("truncated");
                        if (x + count > W) return bad("scanline " + std::to_string(y) + ": run overruns the row");
                        for (size_t k = 0; k < count; k++) row[4 * (x + k) + c] = b[p];
                        p++;
                    } else {
                        if (count == 0 || x + count > W) return bad("scanline " + std::to_string(y) + ": bad literal span");
                        if (p + count > n) return bad("truncated");
                        for (size_t k = 0; k < count; k++) row[4 * (x + k) + c] = b[p + k];
                        p += count;
                    }
                    x += count;
                }
        } else {
            if (p + 4 * (size_t)W > n) return bad("truncated");
            memcpy(row.data(), b + p, 4 * (size_t)W);
            p += 4 * (size_t)W;
        }
        float* out = texels + y * W * 3;
        for (size_t x = 0; x < W; x++) {
            const int e = row[4 * x + 3];
            for (int c = 0; c < 3; c++) out[3 * x + c] = e == 0 ? 0.0f : (float)std::ldexp((double)row[4 * x + c] + 0.5, e - 136);
        }
    }
    return RM_OK;
}

int rm_load_hdr(const char* path, size_t* width, size_t* height, float* texels) {
    if (!path || !width || !height) return fail(RM_ERR_INVALID_ARGUMENT, "rm_load_hdr: null argument");
    std::ifstream f(path, std::ios::binary);
    if (!f) return fail(RM_ERR_IO, std::string("cannot read ") + path);
    std::string buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    if (f.bad()) return fail(RM_ERR_IO, std::string("cannot read ") + path);
    return decode_hdr(buf, path, width, height, texels);
}

size_t rm_tile_layout(const rm_settings* s, size_t* rects, size_t capacity) {
    if (!s) return 0;
    std::vector<TileRect> t = tile_layout(s->camera_settings.backbuffer_width, s->camera_settings.backbuffer_height, s->tile_size[0], s->tile_size[1]);
    for (size_t i = 0; i < t.size() && i < capacity && rects; i++) {
        rects[4 * i] = t[i].left; rects[4 * i + 1] = t[i].top; rects[4 * i + 2] = t[i].width; rects[4 * i + 3] = t[i].height;
    }
    return t.size();
}

// image.save("output.png")                               cli_old/src/main.rs:194-197
// 8-bit RGB, no interlace, filter 0 on every row, zlib stream of stored (uncompressed) deflate blocks.
int rm_write_png(const char* path, const uint8_t* rgb8, size_t width, size_t height) {
    if (!path || (!rgb8 && width != 0 && height != 0)) return fail(RM_ERR_INVALID_ARGUMENT, "rm_write_png: null argument");
    if (width == 0 || height == 0 || width > 0x7fffffffull || height > 0x7fffffffull) return fail(RM_ERR_INVALID_ARGUMENT, "rm_write_png: bad image size");
    static uint32_t table[256];
    static bool have_table = false;
    if (!have_table) {
        for (uint32_t i = 0; i < 256; i++) {
            uint32_t c = i;
            for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
            table[i] = c;
        }
        have_table = true;
    }
    auto crc = [&](const uint8_t* p, size_t n, uint32_t c) { for (size_t i = 0; i < n; i++) c = table[(c ^ p[i]) & 0xff] ^ (c >> 8); return c; };
    auto be32 = [](uint8_t* p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; };
    FILE* f = fopen(path, "wb");
    if (!f) return fail(RM_ERR_IO, std::string("cannot write ") + path);
    bool ok = true;
    auto chunk = [&](const char* type, const uint8_t* data, size_t n) {
        uint8_t hdr[8];
        be32(hdr, (uint32_t)n);
        memcpy(hdr + 4, type, 4);
        uint32_t c = crc(hdr + 4, 4, 0xffffffffu);
        c = crc(data, n, c) ^ 0xffffffffu;
        uint8_t tail[4];
        be32(tail, c);
        ok = ok && fwrite(hdr, 1, 8, f) == 8 && (n == 0 || fwrite(data, 1, n, f) == n) && fwrite(tail, 1, 4, f) == 4;
    };
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    ok = fwrite(sig, 1, 8, f) == 8;
    uint8_t ihdr[13];
    be32(ihdr, (uint32_t)width); be32(ihdr + 4, (uint32_t)height);
    ihdr[8] = 8; ihdr[9] = 2; ihdr[10] = 0; ihdr[11] = 0; ihdr[12] = 0;
    chunk("IHDR", ihdr, 13);
    // raw scanlines: filter byte 0 + 3*width bytes
    const size_t row = 1 + 3 * width, raw_n = row * height;
    std::vector<uint8_t> z;
    try {
        z.reserve(raw_n + raw_n / 65535 * 5 + 16);
        z.push_back(0x78); z.push_back(0x01);
        uint32_t a = 1, b = 0;                                  // Adler-32 of the raw data
        std::vector<uint8_t> raw(raw_n);
        for (size_t y = 0; y < height; y++) { raw[y * row] = 0; memcpy(&raw[y * row + 1], rgb8 + y * 3 * width, 3 * width); }
        for (size_t i = 0; i < raw_n; i++) { a = (a + raw[i]) % 65521u; b = (b + a) % 65521u; }
        for (size_t off = 0; off < raw_n; off += 65535) {
            const size_t n = std::min<size_t>(65535, raw_n - off);
            z.push_back(off + n == raw_n ? 1 : 0);
            z.push_back((uint8_t)(n & 0xff)); z.push_back((uint8_t)(n >> 8));
            z.push_back((uint8_t)(~n & 0xff)); z.push_back((uint8_t)((~n >> 8) & 0xff));
            z.insert(z.end(), raw.begin() + (long)off, raw.begin() + (long)(off + n));
        }
        uint8_t ad[4];
        be32(ad, (b << 16) | a);
        z.insert(z.end(), ad, ad + 4);
    } catch (const std::bad_alloc&) {
        fclose(f);
        return fail(RM_ERR_OUT_OF_MEMORY, "out of memory while encoding the PNG");
    }
    chunk("IDAT", z.data(), z.size());
    chunk("IEND", nullptr, 0);
    ok = (fclose(f) == 0) && ok;
    return ok ? RM_OK : fail(RM_ERR_IO, std::string("short write to ") + path);
}

void rm_tile_free(rm_tile* tile) {
    if (tile && tile->data) { free(tile->data); tile->data = nullptr; }
}

}  // extern "C"
