// raymond_oracle.cpp — CPU ORACLE (test infrastructure, NOT product code).
//
// A line-by-line C++17/f64 restatement of the reference's (Nyrox/raymond) path-
// tracing hot path, used only as the checker in tests/, __graft_entry__.smoke()
// and as the timed CPU baseline of bench.py.  Nothing under raymond_b200/ links,
// loads or calls it.
//
// PARITY UNPINNED: the reference ships no tests, golden vectors or fixtures for
// this path (SURVEY.md §4, §8c) and cannot be built here (no rustc/cargo; the
// arithmetic additionally lives in the un-vendored crates cgmath 0.17, rand 0.6,
// num-traits, versions unpinned because Cargo.lock is git-ignored).  This file
// therefore follows the cited reference lines literally — quirks included
// (SURVEY.md Appendix A) — and restates the third-party semantics from their
// published definitions (Appendix B): cgmath `dot` = (x*x' + y*y') + z*z',
// `normalize` = v * (1/sqrt(dot)), `cast` = range-checked truncation toward
// zero, f64::min/max = NaN-ignoring.  It is anchored by (tests/test_oracle_*.py):
// the reference's own rendered output examples/ReflectiveSpheres.png (block means
// committed under tests/golden/), an independent pure-Python restatement of the
// intersection code, brute-force Mesh::intersects cross-checks and the known
// answers of SURVEY.md Appendix C.
//
// Build: g++ -O2 -ffp-contract=off (rustc never contracts a*b+c into an FMA).
//
// Deviation from the as-is snapshot, shared with the product and documented in
// DESIGN.md: the RNG.  The reference draws rand::random::<f64>() from an
// OS-seeded thread-local generator (never reproducible); the oracle draws the
// same uniforms from a counter-based Philox4x32-10 stream keyed by
// (seed; pixel, sample, depth, draw index) so that a CUDA render can be compared
// sample-for-sample.  All citations are relative to the reference checkout.
//
// The f32-draw mode (bit 1 of rmo_render's flags) exists only to give the product's f32 shading mode
// (RM_PRECISION_F32_SHADING) a same-stream reference: the shading draws of depth >= 1 are that mode's 23-bit uniforms
// instead of the 52-bit ones, and everything else, the arithmetic included, stays this file's f64 restatement.

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <fstream>
#include <memory>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

namespace {

// ---------------------------------------------------------------- math (cgmath 0.17 semantics)

constexpr double PI = 3.14159265358979323846;          // core/src/math.rs:19
constexpr double F_MAX = 1.7976931348623157e308;       // core/src/math.rs:20

struct V3 {
    double x, y, z;
    double& operator[](int i) { return i == 0 ? x : (i == 1 ? y : z); }
    double operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
};
struct V2 { double x, y; };

inline V3 v3(double x, double y, double z) { return V3{x, y, z}; }
inline V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
inline V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
inline V3 operator-(V3 a) { return v3(-a.x, -a.y, -a.z); }
inline V3 operator*(V3 a, double s) { return v3(a.x * s, a.y * s, a.z * s); }
inline V3 operator*(double s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
inline V3 operator/(V3 a, double s) { return v3(a.x / s, a.y / s, a.z / s); }
inline V3 operator/(double s, V3 a) { return v3(s / a.x, s / a.y, s / a.z); }
inline V3 mul_ew(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
inline V3 div_ew(V3 a, V3 b) { return v3(a.x / b.x, a.y / b.y, a.z / b.z); }
// Vector3::dot = mul_element_wise(..).sum() = (x + y) + z
inline double dot(V3 a, V3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
inline V3 cross(V3 a, V3 b) {
    return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
// InnerSpace::normalize = self * (1 / magnitude)
inline V3 normalize(V3 a) { return a * (1.0 / std::sqrt(dot(a, a))); }
// MetricSpace::distance = sqrt((other - self).magnitude2())
inline double distance(V3 a, V3 b) { V3 d = b - a; return std::sqrt(dot(d, d)); }
// Matrix3::from_cols(c0,c1,c2) * v = c0*v.x + c1*v.y + c2*v.z
inline V3 mat_mul(V3 c0, V3 c1, V3 c2, V3 v) { return (c0 * v.x + c1 * v.y) + c2 * v.z; }
// f64::signum: 1.0 for +0.0 and positives, -1.0 for -0.0 and negatives, NaN for NaN
inline double signum(double a) { return std::isnan(a) ? a : (std::signbit(a) ? -1.0 : 1.0); }
// num_traits NumCast f64 -> i32 / usize: Some(trunc) iff MIN-1 < x < MAX+1
inline bool cast_i32(double a, int32_t* out) {
    if (a > -2147483649.0 && a < 2147483648.0) { *out = (int32_t)a; return true; }
    return false;
}
inline bool cast_usize(double a, uint64_t* out) {
    if (a > -1.0 && a < 18446744073709551616.0) { *out = (uint64_t)a; return true; }
    return false;
}
// Rust `x as usize`: saturating, NaN -> 0
inline uint64_t as_usize(double a) {
    if (!(a > 0.0)) return 0;
    if (a >= 18446744073709551616.0) return UINT64_MAX;
    return (uint64_t)a;
}

// ---------------------------------------------------------------- geometry types

struct Ray { V3 origin, direction; };                    // geometry/mod.rs:37-41
struct Hit { double distance; uint64_t subobject_index; }; // geometry/mod.rs:12-17 (the Ray copy is implicit)

struct Vertex { V3 position, normal; V2 uv; V3 tangent; };  // vertex.rs:5-10
struct Triangle { Vertex v0, v1, v2; };                  // triangle.rs:8
static_assert(sizeof(Triangle) == 264, "reference Triangle layout");
struct AABB { V3 min, max; };                            // aabb.rs:4-7

struct Counters {
    uint64_t rays = 0;            // Scene::intersect evaluations
    uint64_t cells = 0;           // grid cells visited (C of SURVEY §8d)
    uint64_t tri_tests = 0;       // Triangle::intersects evaluations (T)
    uint64_t grid_hits = 0;       // AccGrid::intersects returning Some
    uint64_t aabb_tests = 0;      // AABB::intersects evaluations from AccGrid
    uint64_t shaded_tri = 0;      // Triangle::get_surface_properties evaluations
    uint64_t nonfinite = 0;
    uint64_t samples = 0;
    void add(const Counters& o) {
        rays += o.rays; cells += o.cells; tri_tests += o.tri_tests; grid_hits += o.grid_hits;
        aabb_tests += o.aabb_tests; shaded_tri += o.shaded_tri; nonfinite += o.nonfinite; samples += o.samples;
    }
};
thread_local Counters tl_counters;

// Sphere::intersects                                     primitives/sphere.rs:11-27
inline bool sphere_intersects(V3 origin, double radius, const Ray& ray, double* t_out) {
    V3 c = origin - ray.origin;
    double t = dot(c, ray.direction);
    V3 q = c - t * ray.direction;
    double p = dot(q, q);
    if (p > radius * radius) return false;
    t -= std::sqrt(radius * radius - p);
    if (t <= 0.0) return false;
    *t_out = t;
    return true;
}
// Sphere::get_surface_properties                         primitives/sphere.rs:31-35
inline V3 sphere_normal(V3 origin, const Ray& ray, double dist) {
    return normalize((ray.origin + ray.direction * dist) - origin);
}

// Plane::intersects                                      primitives/plane.rs:11-24
inline bool plane_intersects(V3 origin, V3 normal, const Ray& ray, double* t_out) {
    double denom = dot(normal, -ray.direction);
    if (denom > 1e-6) {
        V3 p0l0 = origin - ray.origin;
        double t = dot(p0l0, -normal) / denom;
        if (t >= 0.0) { *t_out = t; return true; }
    }
    return false;
}

// AABB::intersects                                       primitives/aabb.rs:10-31
inline bool aabb_intersects(const AABB& b, const Ray& ray, double* tmin_out) {
    V3 inv = 1.0 / ray.direction;
    double t1 = (b.min[0] - ray.origin[0]) * inv[0];
    double t2 = (b.max[0] - ray.origin[0]) * inv[0];
    double tmin = std::fmin(t1, t2);
    double tmax = std::fmax(t1, t2);
    for (int i = 1; i < 3; i++) {
        t1 = (b.min[i] - ray.origin[i]) * inv[i];
        t2 = (b.max[i] - ray.origin[i]) * inv[i];
        tmin = std::fmax(tmin, std::fmin(t1, t2));
        tmax = std::fmin(tmax, std::fmax(t1, t2));
    }
    if (!(tmax > std::fmax(tmin, 0.0))) return false;
    *tmin_out = tmin;
    return true;
}

// Triangle::intersects (Moller-Trumbore)                 primitives/triangle.rs:11-44
inline bool triangle_intersects(const Triangle& tri, const Ray& ray, double* t_out) {
    const double EPSILON = 0.00000001;
    V3 vertex0 = tri.v0.position, vertex1 = tri.v1.position, vertex2 = tri.v2.position;
    V3 edge1 = vertex1 - vertex0;
    V3 edge2 = vertex2 - vertex0;
    V3 h = cross(ray.direction, edge2);
    double a = dot(edge1, h);
    if (a < EPSILON && a > -EPSILON) return false;
    double f = 1.0 / a;
    V3 s = ray.origin - vertex0;
    double u = f * dot(s, h);
    if (u < 0.0 || u > 1.0) return false;
    V3 q = cross(s, edge1);
    double v = f * dot(ray.direction, q);
    if (v < 0.0 || u + v > 1.0) return false;
    double t = f * dot(edge2, q);
    if (t > EPSILON) { *t_out = t; return true; }
    return false;
}

// Triangle::get_surface_properties (Heron-area barycentrics)   triangle.rs:47-68
inline double heron_area(V3 a, V3 b, V3 c) {
    double ab = distance(a, b);
    double ac = distance(a, c);
    double bc = distance(b, c);
    double s = (ab + ac + bc) / 2.0;
    return std::sqrt(s * (s - ab) * (s - ac) * (s - bc));
}
inline V3 triangle_normal(const Triangle& tri, const Ray& ray, double dist) {
    V3 position = ray.origin + ray.direction * dist;
    double abc = heron_area(tri.v0.position, tri.v1.position, tri.v2.position);
    double abp = heron_area(tri.v0.position, tri.v1.position, position);
    double bcp = heron_area(tri.v0.position, tri.v2.position, position);
    double ba = abp / abc;
    double bb = bcp / abc;
    double bc = 1.0 - (ba + bb);
    V3 normal = (tri.v2.normal * ba) + (tri.v1.normal * bb) + (tri.v0.normal * bc);
    return normalize(normal);
}

// Triangle::find_bounds                                   triangle.rs:70-84
inline AABB triangle_bounds(const Triangle& t) {
    V3 mn = v3(125125.0, 1251251.0, 12512512.0);
    V3 mx = v3(-123125.0, -125123.0, -512123.0);
    for (int i = 0; i < 3; i++) {
        mn[i] = std::fmin(mn[i], t.v0.position[i]);
        mn[i] = std::fmin(mn[i], t.v1.position[i]);
        mn[i] = std::fmin(mn[i], t.v2.position[i]);
        mx[i] = std::fmax(mx[i], t.v0.position[i]);
        mx[i] = std::fmax(mx[i], t.v1.position[i]);
        mx[i] = std::fmax(mx[i], t.v2.position[i]);
    }
    return AABB{mn, mx};
}

// ---------------------------------------------------------------- Mesh

struct Mesh {                                              // mesh.rs:10-13
    std::vector<Triangle> triangles;
    AABB bounding_box;
};

// Mesh::find_mesh_bounds                                  mesh.rs:123-140
AABB find_mesh_bounds(const std::vector<Triangle>& tris) {
    V3 mn = v3(125125.0, 1251251.0, 12512512.0);
    V3 mx = v3(-123125.0, -125123.0, -512123.0);
    for (const Triangle& tri : tris) {
        for (int i = 0; i < 3; i++) {
            mn[i] = std::fmin(mn[i], tri.v0.position[i]);
            mn[i] = std::fmin(mn[i], tri.v1.position[i]);
            mn[i] = std::fmin(mn[i], tri.v2.position[i]);
            mx[i] = std::fmax(mx[i], tri.v0.position[i]);
            mx[i] = std::fmax(mx[i], tri.v1.position[i]);
            mx[i] = std::fmax(mx[i], tri.v2.position[i]);
        }
    }
    return AABB{mn, mx};
}

// Mesh::bake_transform                                    mesh.rs:48-56
void bake_transform(Mesh& m, V3 translate) {
    for (Triangle& t : m.triangles) {
        t.v0.position = t.v0.position + translate;
        t.v1.position = t.v1.position + translate;
        t.v2.position = t.v2.position + translate;
    }
    m.bounding_box = find_mesh_bounds(m.triangles);
}

// Mesh::intersects (brute force; not reachable from Scene)     mesh.rs:23-42
bool mesh_intersects(const Mesh& m, const Ray& ray, Hit* out) {
    double tmin;
    if (!aabb_intersects(m.bounding_box, ray, &tmin)) return false;
    double closest = F_MAX;
    bool any = false;
    for (size_t i = 0; i < m.triangles.size(); i++) {
        double d;
        if (triangle_intersects(m.triangles[i], ray, &d)) {
            if (d < closest) { closest = d; *out = Hit{closest, (uint64_t)i}; any = true; }
        }
    }
    return any;
}

// Vertex::calculate_tangent                               vertex.rs:13-27
V3 calculate_tangent(const Vertex& x, const Vertex& y, const Vertex& z) {
    V3 edge1 = y.position - x.position;
    V3 edge2 = z.position - x.position;
    V2 uv1{y.uv.x - x.uv.x, y.uv.y - x.uv.y};
    V2 uv2{z.uv.x - x.uv.x, z.uv.y - x.uv.y};
    double f = 1.0 / (uv1.x * uv2.y - uv2.x * uv1.y);
    V3 tangent = v3(0.0, 0.0, 0.0);
    tangent.x = f * (uv2.y * edge1.x - uv1.y * edge2.x);
    tangent.y = f * (uv2.y * edge1.y - uv1.y * edge2.y);
    tangent.z = f * (uv2.y * edge1.z - uv1.y * edge2.z);
    return normalize(tangent);
}

std::vector<std::string> split_ws(const std::string& line) {
    std::vector<std::string> out;
    std::istringstream is(line);
    std::string tok;
    while (is >> tok) out.push_back(tok);
    return out;
}

// Mesh::load_ply                                          mesh.rs:58-121
// Returns 0, or -2 (io) / -3 (a Rust unwrap()/index panic while parsing).
int load_ply(const char* path, Mesh* out) {
    std::ifstream f(path, std::ios::binary);
    if (!f) return -2;
    std::stringstream ss; ss << f.rdbuf();
    std::string buffer = ss.str();
    // str::lines(): split on '\n', strip a trailing '\r', no trailing empty line
    std::vector<std::string> lines;
    {
        size_t pos = 0;
        while (pos < buffer.size()) {
            size_t e = buffer.find('\n', pos);
            if (e == std::string::npos) e = buffer.size();
            std::string l = buffer.substr(pos, e - pos);
            if (!l.empty() && l.back() == '\r') l.pop_back();
            lines.push_back(l);
            pos = e + 1;
        }
    }
    size_t li = 0;
    size_t vertex_capacity = 0;
    std::vector<Vertex> vertices;
    std::vector<Triangle> faces;
    // header                                              mesh.rs:66-77
    while (li < lines.size()) {
        std::vector<std::string> tokens = split_ws(lines[li++]);
        if (tokens.empty()) return -3;                      // tokens.next().unwrap()
        if (tokens[0] == "element") {
            if (tokens.size() < 2) return -3;
            if (tokens[1] == "vertex") {
                if (tokens.size() < 3) return -3;
                char* end = nullptr;
                unsigned long long n = std::strtoull(tokens[2].c_str(), &end, 10);
                if (*end != 0) return -3;
                vertex_capacity = (size_t)n;               // reserve_exact
            }
        } else if (tokens[0] == "end_header") {
            break;
        }
    }
    // vertices                                            mesh.rs:80-90
    vertices.reserve(vertex_capacity);
    for (size_t i = 0; i < vertex_capacity; i++) {
        if (li >= lines.size()) return -3;                  // lines.next().unwrap()
        std::vector<std::string> tokens = split_ws(lines[li++]);
        std::vector<double> values;
        for (const std::string& t : tokens) {
            char* end = nullptr;
            double v = std::strtod(t.c_str(), &end);
            if (end == t.c_str() || *end != 0) return -3;
            values.push_back(v);
        }
        if (values.size() < 6) return -3;                   // values[5] out of bounds
        Vertex v;
        v.position = v3(values[0], values[1], values[2]);
        v.normal = v3(values[3], values[4], values[5]);
        v.uv = V2{values.size() > 6 ? values[6] : 0.0, values.size() > 7 ? values[7] : 0.0};
        v.tangent = v3(0.0, 0.0, 0.0);
        vertices.push_back(v);
    }
    // faces                                               mesh.rs:93-118
    while (li < lines.size()) {
        std::vector<std::string> tokens = split_ws(lines[li++]);
        std::vector<uint32_t> values;
        for (const std::string& t : tokens) {
            char* end = nullptr;
            if (t.empty() || t[0] == '-') return -3;
            unsigned long long v = std::strtoull(t.c_str(), &end, 10);
            if (end == t.c_str() || *end != 0 || v > 0xFFFFFFFFull) return -3;
            values.push_back((uint32_t)v);
        }
        if (values.empty()) return -3;                      // values[0]
        if (values[0] == 3) {
            if (values.size() < 4) return -3;
            uint32_t face[3] = {values[1], values[2], values[3]};
            for (int k = 0; k < 3; k++) if (face[k] >= vertices.size()) return -3;
            V3 tangent = calculate_tangent(vertices[face[0]], vertices[face[1]], vertices[face[2]]);
            vertices[face[0]].tangent = tangent;
            vertices[face[1]].tangent = tangent;
            vertices[face[2]].tangent = tangent;
            faces.push_back(Triangle{vertices[values[1]], vertices[values[2]], vertices[values[3]]});
        }
    }
    out->triangles = std::move(faces);
    out->bounding_box = find_mesh_bounds(out->triangles);   // Mesh::new  mesh.rs:16-21
    return 0;
}

// ---------------------------------------------------------------- AccGrid

const double GRID_DENSITY_BIAS = 3.0;                       // acc_grid.rs:4

// estimate_grid_resolution                                acc_grid.rs:6-17
void estimate_grid_resolution(const AABB& bounds, size_t triangle_count, uint64_t res[3]) {
    V3 size = bounds.max - bounds.min;
    double volume = std::fabs(size.x * size.y * size.z);
    double triangle_density = std::pow((GRID_DENSITY_BIAS * (double)triangle_count) / volume, 1.0 / 3.0);
    res[0] = as_usize(std::fabs(size.x) * triangle_density);
    res[1] = as_usize(std::fabs(size.y) * triangle_density);
    res[2] = as_usize(std::fabs(size.z) * triangle_density);
}

struct AccGrid {                                            // acc_grid.rs:27-33
    std::vector<uint64_t> cells;          // Cell(usize): offset into mapping_table
    Mesh mesh;
    std::vector<uint64_t> mapping_table;  // per cell: [count, tri idx ...]
    uint64_t resolution[3];
    V3 cell_size;
};

// AccGrid::build_from_mesh                                acc_grid.rs:36-83
// Returns 0, -4 (Vec index OOB at :61), -5 (zero resolution), -6 (cast failure :47/:51).
int build_from_mesh(Mesh&& mesh, AccGrid* g) {
    uint64_t grid_res[3];
    estimate_grid_resolution(mesh.bounding_box, mesh.triangles.size(), grid_res);
    if (grid_res[0] == 0 || grid_res[1] == 0 || grid_res[2] == 0) return -5;   // `grid_res[i] - 1` underflows
    V3 cell_size = div_ew(mesh.bounding_box.max - mesh.bounding_box.min,
                          v3((double)grid_res[0], (double)grid_res[1], (double)grid_res[2]));
    uint64_t n_cells = grid_res[0] * grid_res[1] * grid_res[2];
    std::vector<std::vector<uint64_t>> naive_cells(n_cells);
    for (size_t index = 0; index < mesh.triangles.size(); index++) {
        AABB bounds = triangle_bounds(mesh.triangles[index]);
        V3 lo = div_ew(bounds.min - mesh.bounding_box.min, cell_size);
        V3 hi = div_ew(bounds.max - mesh.bounding_box.min, cell_size);
        uint64_t cell_min[3], cell_max[3];
        for (int i = 0; i < 3; i++) {
            if (!cast_usize(lo[i], &cell_min[i])) return -6;
            if (!cast_usize(hi[i], &cell_max[i])) return -6;
        }
        for (int i = 0; i < 3; i++) {
            cell_min[i] = std::min(std::max(cell_min[i], (uint64_t)0), grid_res[i] - 1);
            cell_max[i] = std::min(std::max(cell_max[i], (uint64_t)0), grid_res[i] - 1);
        }
        for (uint64_t z = cell_min[2]; z <= cell_max[2]; z++)
            for (uint64_t y = cell_min[1]; y <= cell_max[1]; y++)
                for (uint64_t x = cell_min[0]; x <= cell_max[0]; x++) {
                    uint64_t idx = x + grid_res[0] * (y + z * grid_res[2]);   // sic: z stride is res.z
                    if (idx >= n_cells) return -4;                             // Vec index panic
                    naive_cells[idx].push_back(index);
                }
    }
    g->cells.clear();
    g->mapping_table.clear();
    g->cells.reserve(n_cells);
    for (const std::vector<uint64_t>& c : naive_cells) {
        g->cells.push_back(g->mapping_table.size());
        g->mapping_table.push_back(c.size());
        for (uint64_t i : c) g->mapping_table.push_back(i);
    }
    g->mesh = std::move(mesh);
    g->resolution[0] = grid_res[0]; g->resolution[1] = grid_res[1]; g->resolution[2] = grid_res[2];
    g->cell_size = cell_size;
    return 0;
}

// AccGrid::intersects                                     acc_grid.rs:89-185
// `*panic` is set when the reference would panic on a failed cast (:94,:98,:102).
bool grid_intersects(const AccGrid& g, const Ray& ray, Hit* out, bool* panic) {
    Counters& cnt = tl_counters;
    cnt.aabb_tests++;
    double outer_t;
    if (!aabb_intersects(g.mesh.bounding_box, ray, &outer_t)) return false;
    V3 outer_hit_position = ray.origin + ray.direction * outer_t;

    V3 start = ray.origin - g.mesh.bounding_box.min;
    int32_t cell[3];
    V3 q = div_ew(start, g.cell_size);
    for (int i = 0; i < 3; i++) if (!cast_i32(q[i], &cell[i])) { *panic = true; return false; }
    if (cell[0] < 0 || cell[1] < 0 || cell[2] < 0) {
        start = outer_hit_position - g.mesh.bounding_box.min;
        q = div_ew(start, g.cell_size);
        for (int i = 0; i < 3; i++) if (!cast_i32(q[i], &cell[i])) { *panic = true; return false; }
    }
    int32_t step[3];
    for (int i = 0; i < 3; i++) if (!cast_i32(signum(ray.direction[i]), &step[i])) { *panic = true; return false; }

    double t_delta_x = (ray.direction.x < 0.0 ? -g.cell_size.x : g.cell_size.x) / ray.direction.x;
    double t_delta_y = (ray.direction.y < 0.0 ? -g.cell_size.y : g.cell_size.y) / ray.direction.y;
    double t_delta_z = (ray.direction.z < 0.0 ? -g.cell_size.z : g.cell_size.z) / ray.direction.z;

    double t_max_x = (((double)(cell[0] + (ray.direction.x < 0.0 ? 0 : 1)) * g.cell_size.x) - start.x) / ray.direction.x;
    double t_max_y = (((double)(cell[1] + (ray.direction.y < 0.0 ? 0 : 1)) * g.cell_size.y) - start.y) / ray.direction.y;
    double t_max_z = (((double)(cell[2] + (ray.direction.z < 0.0 ? 0 : 1)) * g.cell_size.z) - start.z) / ray.direction.z;

    const uint64_t rx = g.resolution[0], ry = g.resolution[1], rz = g.resolution[2];
    for (;;) {
        // `as usize` of a non-negative i32; wrapping arithmetic as in a release build
        uint64_t x = (uint64_t)(int64_t)cell[0], y = (uint64_t)(int64_t)cell[1], z = (uint64_t)(int64_t)cell[2];
        uint64_t idx = x + rx * (y + z * rz);
        if (idx >= g.cells.size()) return false;
        cnt.cells++;
        uint64_t cell_off = g.cells[idx];
        uint64_t count = g.mapping_table[cell_off];
        double closest = 5712515.0;
        bool have = false;
        Hit closest_hit{0.0, 0};
        for (uint64_t i = 1; i <= count; i++) {
            const Triangle& tri = g.mesh.triangles[g.mapping_table[cell_off + i]];
            cnt.tri_tests++;
            double d;
            if (triangle_intersects(tri, ray, &d)) {
                if (d < closest) {
                    closest = d;
                    closest_hit = Hit{d, g.mapping_table[cell_off + i]};
                    have = true;
                }
            }
        }
        if (have) { *out = closest_hit; cnt.grid_hits++; return true; }

        if (t_max_x < t_max_y) {
            if (t_max_x < t_max_z) {
                cell[0] += step[0];
                if (cell[0] >= (int32_t)rx || cell[0] < 0) return false;
                t_max_x += t_delta_x;
            } else {
                cell[2] += step[2];
                if (cell[2] >= (int32_t)rz || cell[2] < 0) return false;
                t_max_z += t_delta_z;
            }
        } else {
            if (t_max_y < t_max_z) {
                cell[1] += step[1];
                if (cell[1] >= (int32_t)ry || cell[1] < 0) return false;
                t_max_y += t_delta_y;
            } else {
                cell[2] += step[2];
                if (cell[2] >= (int32_t)rz || cell[2] < 0) return false;
                t_max_z += t_delta_z;
            }
        }
    }
}

// ---------------------------------------------------------------- Scene

enum GeometryKind { GEO_PLANE = 0, GEO_SPHERE = 1, GEO_GRID = 2 };      // scene.rs:9-13
enum MaterialKind { MAT_DIFFUSE = 0, MAT_METAL = 1, MAT_EMISSION = 2 };  // lib.rs:21-26

struct Material { int kind; V3 a; V3 b; double p0, p1; };

struct Object {                                             // scene.rs:33-37
    int geometry;
    V3 origin; V3 normal; double radius;
    std::shared_ptr<AccGrid> grid;                          // Arc<AccGrid>
    Material material;
};

struct Scene { std::vector<Object> objects; };              // scene.rs:42-45

// Scene::intersect                                        scene.rs:54-74
bool scene_intersect(const Scene& scene, const Ray& ray, size_t* object_out, Hit* hit_out) {
    tl_counters.rays++;
    double closest_distance = F_MAX;
    bool any = false;
    for (size_t i = 0; i < scene.objects.size(); i++) {
        const Object& o = scene.objects[i];
        Hit hit{0.0, 0};
        bool got = false;
        switch (o.geometry) {                               // Geometry::intersects  scene.rs:16-22
            case GEO_PLANE: got = plane_intersects(o.origin, o.normal, ray, &hit.distance); break;
            case GEO_SPHERE: got = sphere_intersects(o.origin, o.radius, ray, &hit.distance); break;
            case GEO_GRID: { bool panic = false; got = grid_intersects(*o.grid, ray, &hit, &panic); break; }
        }
        if (got) {
            if (hit.distance < closest_distance) {
                closest_distance = hit.distance;
                *object_out = i;
                *hit_out = hit;
                any = true;
            }
        }
    }
    return any;
}

// Geometry::get_surface_properties                        scene.rs:24-30
V3 surface_normal(const Object& o, const Ray& ray, const Hit& hit) {
    switch (o.geometry) {
        case GEO_PLANE: return o.normal;                                       // plane.rs:28-32
        case GEO_SPHERE: return sphere_normal(o.origin, ray, hit.distance);
        default:
            tl_counters.shaded_tri++;
            return triangle_normal(o.grid->mesh.triangles[hit.subobject_index], ray, hit.distance);  // acc_grid.rs:85-87
    }
}

// ---------------------------------------------------------------- RNG (documented deviation)

struct Philox {
    static inline void round(uint32_t c[4], uint32_t k0, uint32_t k1) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    }
    static inline void block(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) {
        uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
        uint32_t c[4] = {c0, c1, c2, c3};
        for (int r = 0; r < 10; r++) {
            round(c, k0, k1);
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
        out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
    }
};
// 52 random bits -> (k + 0.5) * 2^-52, strictly inside (0, 1)
inline double u52(uint32_t hi, uint32_t lo) {
    uint64_t bits = ((uint64_t)hi << 32) | lo;
    return ((double)(bits >> 12) + 0.5) * (1.0 / 4503599627370496.0);
}
// 23 random bits -> (k + 0.5) * 2^-23, the f32 shading mode's uniform; exact as a double
inline double u23(uint32_t x) {
    return ((double)(x >> 9) + 0.5) * (1.0 / 8388608.0);
}
// Stands in for rand::random::<f64>(): draw number `index` of (pixel, sample, depth).
// f32_draws: the shading draws (depth >= 1) are those of the product's f32 shading mode, all three from one Philox block:
// the lobe choice from word 0, the next draw (diffuse theta / specular phi) from word 2, the last (diffuse phi / GGX theta)
// from word 1.  Camera draws (depth 0) are the 52-bit ones in both modes.
struct Sampler {
    uint64_t seed; uint32_t pixel; uint32_t sample; bool f32_draws = false;
    double draw(uint32_t depth, uint32_t index) const {
        uint32_t w[4];
        if (f32_draws && depth >= 1) {
            Philox::block(seed, pixel, sample, depth, 0, w);
            return u23(w[index == 0 ? 0 : (index == 1 ? 2 : 1)]);
        }
        Philox::block(seed, pixel, sample, depth, index >> 1, w);
        return (index & 1) ? u52(w[2], w[3]) : u52(w[0], w[1]);
    }
};

// ---------------------------------------------------------------- integrator (src/trace.rs)

struct CameraSettings {                                     // src/trace.rs:32-40
    size_t backbuffer_width, backbuffer_height;
    double fov_vert; V3 position; double focal_length, aperture_radius;
};
struct Settings {                                           // src/trace.rs:42-55
    size_t worker_count; CameraSettings camera_settings; size_t sample_count;
    size_t samples_per_iteration; size_t tile_size[2]; size_t bounce_limit;
};
struct TraceContext { const Scene* scene; const Settings* settings; };   // src/trace.rs:57-60

inline double lerp(double mn, double mx, double a) { return mn + a * (mx - mn); }          // :392-394
inline V3 lerp_vec(V3 mn, V3 mx, double a) { return v3(lerp(mn.x, mx.x, a), lerp(mn.y, mx.y, a), lerp(mn.z, mx.z, a)); }  // :388-390

// ggx_distribution                                        src/trace.rs:362-370
double ggx_distribution(V3 n, V3 h, double roughness) {
    double a2 = roughness * roughness;
    double NdotH = dot(n, h);
    double nominator = a2;
    double denominator = std::pow(NdotH, 2.0) * (a2 - 1.0) + 1.0;
    denominator = std::fmax(PI * denominator * denominator, 1e-7);
    return nominator / denominator;
}
// geometry_schlick_ggx                                    src/trace.rs:372-378
double geometry_schlick_ggx(V3 n, V3 v, double r) {
    double numerator = std::fmax(dot(n, v), 0.0);
    double k = (r * r) / 8.0;
    double denominator = numerator * (1.0 - k) + k;
    return numerator / denominator;
}
// geometry_smith                                          src/trace.rs:380-382
double geometry_smith(V3 n, V3 v, V3 l, double r) { return geometry_schlick_ggx(n, v, r) * geometry_schlick_ggx(n, l, r); }
// fresnel_schlick                                         src/trace.rs:384-386
V3 fresnel_schlick(double cos_theta, V3 F0) { return F0 + (v3(1.0, 1.0, 1.0) - F0) * std::pow(1.0 - cos_theta, 5.0); }
// create_coordinate_system_of_n                           src/trace.rs:408-416
void create_coordinate_system_of_n(V3 n, V3* t, V3* b) {
    double sign = n.z > 0.0 ? 1.0 : -1.0;
    double a = -1.0 / (sign + n.z);
    double bb = n.x * n.y * a;
    *t = v3(1.0 + sign * n.x * n.x * a, sign * bb, -sign * n.x);
    *b = v3(bb, sign + n.y * n.y * a, -n.y);
}
// uniform_sample_hemisphere                               src/trace.rs:396-406
void uniform_sample_hemisphere(double r1, double r2, V3* cartesian, double* pdf) {
    double theta = std::acos(std::sqrt(r1));
    double phi = 2.0 * PI * r2;
    *pdf = std::sqrt(r1);
    *cartesian = v3(std::sin(theta) * std::cos(phi), std::cos(theta), std::sin(theta) * std::sin(phi));
}
// importance_sample_ggx                                   src/trace.rs:286-296
V3 importance_sample_ggx(V3 reflect, double roughness, double r1, double r2) {
    double a = roughness * roughness;
    double phi = 2.0 * PI * r1;
    double theta = a * std::sqrt(r2 / (1.0 - r2));
    V3 h = v3(std::sin(theta) * std::cos(phi), std::cos(theta), std::sin(theta) * std::sin(phi));
    V3 tangent, bitangent;
    create_coordinate_system_of_n(reflect, &tangent, &bitangent);
    return normalize(mat_mul(tangent, reflect, bitangent, h));
}

// trace                                                   src/trace.rs:232-320
V3 trace(const Ray& ray, const TraceContext& ctx, size_t depth, const Sampler& rng) {
    const Settings& settings = *ctx.settings;
    if (depth > settings.bounce_limit) return v3(0.0, 0.0, 0.0);

    size_t oi; Hit hit;
    if (!scene_intersect(*ctx.scene, ray, &oi, &hit)) return v3(0.0, 0.0, 0.0);
    const Object& object = ctx.scene->objects[oi];
    V3 normal = surface_normal(object, ray, hit);
    V3 fragment_position = ray.origin + ray.direction * hit.distance;
    V3 material_color; double material_roughness, material_metalness;
    switch (object.material.kind) {
        case MAT_DIFFUSE: material_color = object.material.a; material_roughness = object.material.p0; material_metalness = 0.0; break;
        case MAT_METAL: material_color = object.material.a; material_roughness = object.material.p0; material_metalness = 1.0; break;
        default: return object.material.a;                  // Emission(e, _, _, _) => return e
    }

    V3 view_dir = normalize(settings.camera_settings.position - fragment_position);
    V3 f0 = v3(0.04, 0.04, 0.04);
    f0 = lerp_vec(f0, material_color, material_metalness);
    double r = rng.draw((uint32_t)depth, 0);                // rand::random::<f64>()  :260
    V3 lc0, lc1;
    create_coordinate_system_of_n(normal, &lc0, &lc1);
    double prob_d = lerp(0.5, 0.0, material_metalness);
    if (r < prob_d) {
        V3 sample; double pdf;
        uniform_sample_hemisphere(rng.draw((uint32_t)depth, 1), rng.draw((uint32_t)depth, 2), &sample, &pdf);
        V3 sample_world = normalize(mat_mul(lc0, normal, lc1, sample));
        V3 radiance = trace(Ray{fragment_position + normal * 0.00001, sample_world}, ctx, depth + 1, rng);
        double cos_theta = std::fmax(dot(normal, sample_world), 0.0);
        V3 halfway = normalize(sample_world + view_dir);
        V3 fresnel = fresnel_schlick(std::fmax(dot(halfway, view_dir), 0.0), f0);
        V3 specular_part = fresnel;
        V3 diffuse_part = v3(1.0, 1.0, 1.0) - specular_part;
        diffuse_part = diffuse_part * (1.0 - material_metalness);
        V3 output = mul_ew(mul_ew(diffuse_part, material_color), radiance) * cos_theta;
        return output / (prob_d * pdf);
    } else {
        V3 reflect = normalize(-view_dir - 2.0 * (-dot(view_dir, normal) * normal));
        V3 sample_world = importance_sample_ggx(reflect, material_roughness, rng.draw((uint32_t)depth, 1), rng.draw((uint32_t)depth, 2));
        V3 radiance = trace(Ray{fragment_position + normal * 0.0001, sample_world}, ctx, depth + 1, rng);
        double cos_theta = dot(normal, sample_world);
        V3 light_dir = normalize(sample_world);
        V3 halfway = normalize(light_dir + view_dir);
        V3 F = fresnel_schlick(dot(halfway, view_dir), f0);
        double D = ggx_distribution(normal, halfway, material_roughness);
        double G = geometry_smith(normal, view_dir, sample_world, material_roughness);
        V3 nominator = D * G * F;
        double denominator = 4.0 * dot(normal, view_dir) * cos_theta + 0.001;
        V3 specular = nominator / denominator;
        V3 output = mul_ew(specular, radiance) * cos_theta;
        double pdf = (D * dot(normal, halfway)) / (4.0 * dot(halfway, view_dir)) + 0.0001;
        return output / (1.0 - prob_d) / pdf;
    }
}

// generate_primary_ray                                    src/trace.rs:322-333
// jx, jy stand for the two rand::random::<f64>() draws (x first).
Ray generate_primary_ray(size_t xi, size_t yi, const CameraSettings& camera, double jx, double jy) {
    double width = (double)camera.backbuffer_width;
    double height = (double)camera.backbuffer_height;
    double aspect = width / height;
    double x = (double)xi + (jx - 0.5);
    double y = (double)yi + (jy - 0.5);
    double px = (2.0 * ((x + 0.5) / width) - 1.0) * std::tan(camera.fov_vert / 2.0 * PI / 180.0) * aspect;
    double py = (1.0 - 2.0 * ((y + 0.5) / height)) * std::tan(camera.fov_vert / 2.0 * PI / 180.0);
    return Ray{camera.position, normalize(v3(px, py, 1.0))};
}

// generate_primary_ray_with_dof                           src/trace.rs:335-360
// (dead code in the snapshot; selected iff aperture_radius > 0 — it never
// terminates for radius 0.)  Rejection round j uses draws 2+2j, 3+2j of depth 0.
Ray generate_primary_ray_with_dof(size_t xi, size_t yi, const CameraSettings& camera, const Sampler& rng) {
    Ray primary = generate_primary_ray(xi, yi, camera, rng.draw(0, 0), rng.draw(0, 1));
    V3 start;
    for (uint32_t j = 0;; j++) {
        double r1 = rng.draw(0, 2 + 2 * j) * 2.0 - 1.0;
        double r2 = rng.draw(0, 3 + 2 * j) * 2.0 - 1.0;
        double ax = camera.position.x + r1 * camera.aperture_radius;
        double ay = camera.position.y + r2 * camera.aperture_radius;
        V3 s = v3(ax, ay, camera.position.z);
        if (distance(s, camera.position) < camera.aperture_radius) { start = s; break; }
    }
    V3 fp_origin = camera.position + v3(0.0, 0.0, 1.0) * camera.focal_length;
    V3 fp_normal = v3(0.0, 0.0, -1.0);
    double t = 0.0;
    plane_intersects(fp_origin, fp_normal, primary, &t);     // .unwrap()
    V3 end = camera.position + t * primary.direction;
    return Ray{start, normalize(end - start)};
}

Ray camera_ray(size_t x, size_t y, const CameraSettings& camera, const Sampler& rng) {
    if (camera.aperture_radius > 0.0) return generate_primary_ray_with_dof(x, y, camera, rng);
    return generate_primary_ray(x, y, camera, rng.draw(0, 0), rng.draw(0, 1));
}

// ---------------------------------------------------------------- render driver

struct Tile {                                               // core/src/tile.rs:6-14
    size_t sample_count, width, height, left, top;
    std::vector<V3> data;
};

// tile split of render_tiled                              src/trace.rs:142-173
std::vector<Tile> split_tiles(const Settings& settings, bool with_data) {
    std::vector<Tile> tiles;
    size_t x = 0, y = 0;
    const size_t W = settings.camera_settings.backbuffer_width, H = settings.camera_settings.backbuffer_height;
    for (;;) {
        size_t max_x = std::min(x + settings.tile_size[0], W);
        size_t max_y = std::min(y + settings.tile_size[1], H);
        size_t width = max_x - x, height = max_y - y;
        Tile t{0, width, height, x, y, {}};
        if (with_data) t.data.assign(width * height, v3(0.0, 0.0, 0.0));
        tiles.push_back(std::move(t));
        y += settings.tile_size[1];
        if (y >= H) { y = 0; x += settings.tile_size[0]; }
        if (x >= W) break;
    }
    return tiles;
}

}  // namespace

// ================================================================= C API (rmo_*)

extern "C" {

struct rmo_mesh { Mesh m; };
struct rmo_grid { std::shared_ptr<AccGrid> g; };
struct rmo_scene { Scene s; };

struct rmo_vec3 { double x, y, z; };
struct rmo_ray { rmo_vec3 origin, direction; };
struct rmo_material { uint32_t kind; uint32_t reserved; rmo_vec3 a; rmo_vec3 b; double p0; double p1; };
struct rmo_camera { size_t width, height; double fov_vert; rmo_vec3 position; double focal_length, aperture_radius; };
struct rmo_settings { size_t worker_count; rmo_camera camera; size_t sample_count; size_t samples_per_iteration; size_t tile_size[2]; size_t bounce_limit; };
struct rmo_counters { uint64_t rays, cells, tri_tests, grid_hits, aabb_tests, shaded_tri, nonfinite, samples; };

static V3 tov(rmo_vec3 v) { return v3(v.x, v.y, v.z); }
static Ray toray(const rmo_ray& r) { return Ray{tov(r.origin), tov(r.direction)}; }
static void export_counters(const Counters& c, rmo_counters* o) {
    if (!o) return;
    o->rays = c.rays; o->cells = c.cells; o->tri_tests = c.tri_tests; o->grid_hits = c.grid_hits;
    o->aabb_tests = c.aabb_tests; o->shaded_tri = c.shaded_tri; o->nonfinite = c.nonfinite; o->samples = c.samples;
}
static Settings tosettings(const rmo_settings& s) {
    Settings o;
    o.worker_count = s.worker_count;
    o.camera_settings = CameraSettings{s.camera.width, s.camera.height, s.camera.fov_vert, tov(s.camera.position), s.camera.focal_length, s.camera.aperture_radius};
    o.sample_count = s.sample_count; o.samples_per_iteration = s.samples_per_iteration;
    o.tile_size[0] = s.tile_size[0]; o.tile_size[1] = s.tile_size[1]; o.bounce_limit = s.bounce_limit;
    return o;
}

rmo_mesh* rmo_mesh_load_ply(const char* path, int* status) {
    rmo_mesh* m = new rmo_mesh();
    int rc = load_ply(path, &m->m);
    if (status) *status = rc;
    if (rc != 0) { delete m; return nullptr; }
    return m;
}
// `tris` is an array of 264-byte reference-layout triangles
rmo_mesh* rmo_mesh_from_triangles(const void* tris, size_t n) {
    rmo_mesh* m = new rmo_mesh();
    m->m.triangles.resize(n);
    if (n) std::memcpy(m->m.triangles.data(), tris, n * sizeof(Triangle));
    m->m.bounding_box = find_mesh_bounds(m->m.triangles);
    return m;
}
void rmo_mesh_translate(rmo_mesh* m, double x, double y, double z) { bake_transform(m->m, v3(x, y, z)); }
size_t rmo_mesh_count(const rmo_mesh* m) { return m->m.triangles.size(); }
void rmo_mesh_bounds(const rmo_mesh* m, double* out6) {
    const AABB& b = m->m.bounding_box;
    out6[0] = b.min.x; out6[1] = b.min.y; out6[2] = b.min.z; out6[3] = b.max.x; out6[4] = b.max.y; out6[5] = b.max.z;
}
void rmo_mesh_triangles(const rmo_mesh* m, void* out) { std::memcpy(out, m->m.triangles.data(), m->m.triangles.size() * sizeof(Triangle)); }
void rmo_mesh_destroy(rmo_mesh* m) { delete m; }
// Mesh::intersects (brute force) on n rays; tri = -1 on a miss
void rmo_mesh_intersect(const rmo_mesh* m, const rmo_ray* rays, size_t n, int64_t* tri, double* t) {
    for (size_t i = 0; i < n; i++) {
        Hit h;
        if (mesh_intersects(m->m, toray(rays[i]), &h)) { tri[i] = (int64_t)h.subobject_index; t[i] = h.distance; }
        else tri[i] = -1;
    }
}

// consumes the mesh's triangles (the Rust call moves the Mesh)
rmo_grid* rmo_grid_build(rmo_mesh* m, int* status) {
    auto g = std::make_shared<AccGrid>();
    int rc = build_from_mesh(std::move(m->m), g.get());
    m->m = Mesh{};
    if (status) *status = rc;
    if (rc != 0) return nullptr;
    return new rmo_grid{g};
}
void rmo_grid_destroy(rmo_grid* g) { delete g; }
void rmo_grid_info(const rmo_grid* g, uint64_t* res3, double* cell_size3, double* bounds6, uint64_t* n_cells, uint64_t* table_len, uint64_t* n_tris) {
    const AccGrid& a = *g->g;
    for (int i = 0; i < 3; i++) { res3[i] = a.resolution[i]; cell_size3[i] = a.cell_size[i]; }
    const AABB& b = a.mesh.bounding_box;
    bounds6[0] = b.min.x; bounds6[1] = b.min.y; bounds6[2] = b.min.z; bounds6[3] = b.max.x; bounds6[4] = b.max.y; bounds6[5] = b.max.z;
    *n_cells = a.cells.size(); *table_len = a.mapping_table.size(); *n_tris = a.mesh.triangles.size();
}
void rmo_grid_tables(const rmo_grid* g, uint64_t* cells, uint64_t* mapping_table) {
    const AccGrid& a = *g->g;
    std::memcpy(cells, a.cells.data(), a.cells.size() * sizeof(uint64_t));
    std::memcpy(mapping_table, a.mapping_table.data(), a.mapping_table.size() * sizeof(uint64_t));
}
// AccGrid::intersects on n rays; tri = -1 miss, -2 the reference would panic
void rmo_grid_intersect(const rmo_grid* g, const rmo_ray* rays, size_t n, int64_t* tri, double* t, rmo_counters* counters) {
    tl_counters = Counters{};
    for (size_t i = 0; i < n; i++) {
        Hit h; bool panic = false;
        if (grid_intersects(*g->g, toray(rays[i]), &h, &panic)) { tri[i] = (int64_t)h.subobject_index; t[i] = h.distance; }
        else tri[i] = panic ? -2 : -1;
    }
    export_counters(tl_counters, counters);
}

rmo_scene* rmo_scene_create() { return new rmo_scene(); }
void rmo_scene_destroy(rmo_scene* s) { delete s; }
static Material tomat(const rmo_material* m) { return Material{(int)m->kind, tov(m->a), tov(m->b), m->p0, m->p1}; }
void rmo_scene_add_sphere(rmo_scene* s, rmo_vec3 origin, double radius, const rmo_material* m) {
    Object o{}; o.geometry = GEO_SPHERE; o.origin = tov(origin); o.radius = radius; o.normal = v3(0, 0, 0); o.material = tomat(m);
    s->s.objects.push_back(o);
}
void rmo_scene_add_plane(rmo_scene* s, rmo_vec3 origin, rmo_vec3 normal, const rmo_material* m) {
    Object o{}; o.geometry = GEO_PLANE; o.origin = tov(origin); o.normal = tov(normal); o.radius = 0; o.material = tomat(m);
    s->s.objects.push_back(o);
}
void rmo_scene_add_grid(rmo_scene* s, const rmo_grid* g, const rmo_material* m) {
    Object o{}; o.geometry = GEO_GRID; o.origin = v3(0, 0, 0); o.normal = v3(0, 0, 0); o.radius = 0; o.grid = g->g; o.material = tomat(m);
    s->s.objects.push_back(o);
}
// Scene::intersect on n rays, optionally with `threads` workers over contiguous ranges
void rmo_scene_intersect(const rmo_scene* s, const rmo_ray* rays, size_t n, int64_t* obj, uint64_t* sub, double* t, rmo_counters* counters, int threads) {
    if (threads < 1) threads = 1;
    std::vector<Counters> per(threads);
    auto work = [&](int k) {
        tl_counters = Counters{};
        size_t lo = n * (size_t)k / threads, hi = n * (size_t)(k + 1) / threads;
        for (size_t i = lo; i < hi; i++) {
            size_t oi; Hit h;
            if (scene_intersect(s->s, toray(rays[i]), &oi, &h)) { obj[i] = (int64_t)oi; if (sub) sub[i] = h.subobject_index; if (t) t[i] = h.distance; }
            else { obj[i] = -1; if (sub) sub[i] = 0; }
        }
        per[k] = tl_counters;
    };
    if (threads == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int k = 0; k < threads; k++) th.emplace_back(work, k);
        for (auto& x : th) x.join();
    }
    Counters total; for (auto& c : per) total.add(c);
    export_counters(total, counters);
}
// surface normal the integrator would use for hit (obj, sub, t) of ray
void rmo_scene_normal(const rmo_scene* s, const rmo_ray* ray, int64_t obj, uint64_t sub, double t, double* out3) {
    V3 n = surface_normal(s->s.objects[(size_t)obj], toray(*ray), Hit{t, sub});
    out3[0] = n.x; out3[1] = n.y; out3[2] = n.z;
}

// generate_primary_ray for every pixel of the frame, row-major.
// jitter: NULL => the jitter term (rand - 0.5) forced to 0 (pixel centres), else W*H*2 uniforms (x, y).
void rmo_primary_rays(const rmo_camera* cam, const double* jitter, rmo_ray* out) {
    CameraSettings c{cam->width, cam->height, cam->fov_vert, tov(cam->position), cam->focal_length, cam->aperture_radius};
    for (size_t y = 0; y < c.backbuffer_height; y++)
        for (size_t x = 0; x < c.backbuffer_width; x++) {
            size_t p = x + y * c.backbuffer_width;
            Ray r = generate_primary_ray(x, y, c, jitter ? jitter[2 * p] : 0.5, jitter ? jitter[2 * p + 1] : 0.5);
            out[p] = rmo_ray{{r.origin.x, r.origin.y, r.origin.z}, {r.direction.x, r.direction.y, r.direction.z}};
        }
}
// the camera ray (DoF included) of (pixel, sample) under the Philox stream
void rmo_camera_rays(const rmo_camera* cam, uint64_t seed, uint32_t sample, rmo_ray* out) {
    CameraSettings c{cam->width, cam->height, cam->fov_vert, tov(cam->position), cam->focal_length, cam->aperture_radius};
    for (size_t y = 0; y < c.backbuffer_height; y++)
        for (size_t x = 0; x < c.backbuffer_width; x++) {
            size_t p = x + y * c.backbuffer_width;
            Ray r = camera_ray(x, y, c, Sampler{seed, (uint32_t)p, sample});
            out[p] = rmo_ray{{r.origin.x, r.origin.y, r.origin.z}, {r.direction.x, r.direction.y, r.direction.z}};
        }
}
// the uniform the product must reproduce: draw `index` of (seed; pixel, sample, depth)
double rmo_rng_draw(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t depth, uint32_t index) {
    return Sampler{seed, pixel, sample}.draw(depth, index);
}
// the same draw of the f32-draw stream (the product's f32 shading mode); index 0..2
double rmo_rng_draw_f32(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t depth, uint32_t index) {
    return Sampler{seed, pixel, sample, true}.draw(depth, index);
}

size_t rmo_tile_layout(const rmo_settings* s, size_t* rects, size_t capacity) {
    Settings st = tosettings(*s);
    std::vector<Tile> tiles = split_tiles(st, false);
    for (size_t i = 0; i < tiles.size() && i < capacity; i++) {
        rects[4 * i] = tiles[i].left; rects[4 * i + 1] = tiles[i].top; rects[4 * i + 2] = tiles[i].width; rects[4 * i + 3] = tiles[i].height;
    }
    return tiles.size();
}

// render_tiled + TaskHandle::await                        src/trace.rs:137-230, 82-113
// As-is structure: worker_count threads pop tiles from a FIFO queue, render ONE
// sample per pixel per pass, push the tile back until sample_count is reached,
// and retire for good the first time they find the queue empty (:189-195).
//   first_sample/sample_stride: global sample index of pass k is first + k*stride
//   flags bit 0: drop (and count) non-finite samples instead of accumulating them
//   flags bit 1: the f32-draw stream (see Sampler)
//   out_sum: W*H*3 running sums (row-major) — divide by sample_count for await()'s output
int rmo_render(const rmo_scene* scene, const rmo_settings* s, uint64_t seed, uint32_t first_sample, uint32_t sample_stride,
               uint32_t flags, double* out_sum, rmo_counters* counters) {
    Settings settings = tosettings(*s);
    const size_t W = settings.camera_settings.backbuffer_width, H = settings.camera_settings.backbuffer_height;
    if (settings.tile_size[0] == 0 || settings.tile_size[1] == 0 || W == 0 || H == 0) return -1;
    std::deque<Tile> queue;
    std::mutex qm;
    for (Tile& t : split_tiles(settings, true)) queue.push_back(std::move(t));
    std::vector<Tile> finished;
    std::mutex fm;
    TraceContext ctx{&scene->s, &settings};
    size_t workers = settings.worker_count ? settings.worker_count : 1;
    std::vector<Counters> per(workers);
    std::vector<std::thread> threads;
    for (size_t w = 0; w < workers; w++) {
        threads.emplace_back([&, w]() {
            tl_counters = Counters{};
            for (;;) {
                Tile tile;
                {
                    std::lock_guard<std::mutex> lk(qm);
                    if (queue.empty()) break;                 // try_pop() == None => thread exits
                    tile = std::move(queue.front());
                    queue.pop_front();
                }
                uint32_t sample = first_sample + (uint32_t)tile.sample_count * sample_stride;
                for (size_t y = tile.top; y < tile.top + tile.height; y++) {
                    for (size_t x = tile.left; x < tile.left + tile.width; x++) {
                        Sampler rng{seed, (uint32_t)(x + y * W), sample, (flags & 2u) != 0};
                        Ray primary = camera_ray(x, y, settings.camera_settings, rng);
                        V3 smp = trace(primary, ctx, 1, rng);
                        tl_counters.samples++;
                        bool finite = std::isfinite(smp.x) && std::isfinite(smp.y) && std::isfinite(smp.z);
                        if (!finite) { tl_counters.nonfinite++; if (flags & 1u) continue; }
                        V3& d = tile.data[(x - tile.left) + (y - tile.top) * tile.width];
                        d = d + smp;
                    }
                }
                tile.sample_count += 1;
                if (tile.sample_count == settings.sample_count) {
                    std::lock_guard<std::mutex> lk(fm);
                    finished.push_back(std::move(tile));      // Message::TileFinished
                } else {
                    std::lock_guard<std::mutex> lk(qm);
                    queue.push_back(std::move(tile));
                }
            }
            per[w] = tl_counters;
        });
    }
    for (auto& t : threads) t.join();
    for (const Tile& tile : finished)
        for (size_t y = 0; y < tile.height; y++)
            for (size_t x = 0; x < tile.width; x++) {
                const V3& v = tile.data[x + y * tile.width];
                double* o = out_sum + 3 * (x + tile.left + (y + tile.top) * W);
                o[0] = v.x; o[1] = v.y; o[2] = v.z;
            }
    Counters total; for (auto& c : per) total.add(c);
    export_counters(total, counters);
    return 0;
}

// radiance of single paths: trace(camera_ray(pixel), depth 1) for listed (pixel, sample) pairs
void rmo_trace_samples(const rmo_scene* scene, const rmo_settings* s, uint64_t seed, const uint32_t* pixels, const uint32_t* samples, size_t n, double* out3) {
    Settings settings = tosettings(*s);
    TraceContext ctx{&scene->s, &settings};
    const size_t W = settings.camera_settings.backbuffer_width;
    for (size_t i = 0; i < n; i++) {
        Sampler rng{seed, pixels[i], samples[i]};
        Ray primary = camera_ray(pixels[i] % W, pixels[i] / W, settings.camera_settings, rng);
        V3 v = trace(primary, ctx, 1, rng);
        out3[3 * i] = v.x; out3[3 * i + 1] = v.y; out3[3 * i + 2] = v.z;
    }
}

}  // extern "C"
