// rm_kernels.cuh — device code of the hot path (sm_100a): data model, the bit-exact f64 intersection
// routines, the counter-based RNG, camera, shading, and the wavefront kernels.
//
// One wavefront stage (= one recursion level of the reference's `trace`, src/trace.rs:232-320) is
// three kernels, so that every warp does one kind of work:
//   k_setup     one thread per ray: [camera ray generation |  queue read], the analytic objects
//               (Sphere / Plane), AABB::intersects + DDA set-up of the grid; rays that enter a grid
//               are appended (ballot/popc compaction) to a traversal queue of 128-byte records
//   k_traverse  persistent warps over the traversal queue: AccGrid::intersects in three warp-uniform phases — lanes
//               walk their ray's DDA four cells ahead to the next occupied cell; the triangle lists of all 32 rays
//               are pooled, a conservative bounding-sphere pre-test drops the candidates the reference is certain
//               to reject, and Triangle::intersects runs on the survivors with full lanes; rays with a hit finish,
//               idle lanes re-fill from the queue in groups
//   k_shade     one thread per ray: surface normal, material, lobe choice, BRDF weight, next ray or
//               delivered radiance; survivors are compacted into the next stage's ray queue.  At the bounce limit in
//               drop mode only the emitter test is left (k_shade<..., LAST>), and k_setup queues no traversal for a ray
//               whose closest hit so far is not an emitter (SetupArgs::emitters_only)
// followed once per batch by k_accumulate (the tile accumulator).
// (Round 2 measured two variations of this pipeline and kept neither — profiles/r2_ab_fusion_binning_f32.log: k_shade fused with
// the next depth's k_setup starves on instruction fetch, 4 000-5 000 SASS instructions, stall_no_instruction 6.4 per issue;
// binning the bounced rays by start cell and direction octant before k_traverse buys 4 % of its time and costs as much.)
//
// Build with -fmad=false: rustc never contracts a*b+c, and every f64 add/mul/div/sqrt below is one
// IEEE operation in the reference's order.  Citations are relative to the reference checkout.
#pragma once

#include <cuda_runtime.h>

#include <cfloat>

#include "rm_internal.hpp"

namespace rm {

// ===================================================================== device data model

constexpr int kMaxObjects = 64;   // objects carried in the kernel parameter block (constant bank)
constexpr int kMaxGrids = 8;
constexpr int kBlock = 256;
// resident blocks per SM the register allocation of each kernel is bounded for (tuning: -DRM_..._BLOCKS_PER_SM=n)
#ifndef RM_SHADE_BLOCKS_PER_SM
#define RM_SHADE_BLOCKS_PER_SM 4
#endif
#ifndef RM_SETUP_BLOCKS_PER_SM
#define RM_SETUP_BLOCKS_PER_SM 4
#endif

// One AccGrid resident in HBM.
//   cells : {first reference, count} per cell            (8 B, one 64-bit load per visited cell)
//   refs  : triangle indices, ascending inside a cell     (4 B per reference)
//   tri   : 96 B per triangle, 32 B aligned, 3 sectors: [v0.xyz v1.x][v1.yz v2.xy][v2.z 0 0 0]
//   sphr  : 16 B per reference (f32 centre + inflated radius of the triangle's bounding sphere), in the order of `refs`, so the
//           candidates of a cell are one contiguous, coalesced read; candidates whose ray line provably misses the sphere
//           skip the reference, the 96-B fetch and the test
//   shd   : 144 B per triangle (v0 v1 v2 n0 n1 n2), read once per shaded hit
//   occ   : 1 bit per cell, set when the cell holds any reference — 64x smaller than `cells`, so the walk
//           through empty cells (most of a ray's cells) is served from L1 instead of one L2 trip per cell
struct DevGrid {
    double bmin[3], bmax[3], cell[3];
    int res[3];
    int pad;
    double diag2;             // squared diagonal of the bounding box (bounds the squared length of any triangle edge)
    double diag;              // ... and the diagonal (bounds the distance between any two points of the box)
    unsigned long long n_cells;
    const uint2* cells;
    const unsigned* occ;
    const unsigned* refs;
    const double* tri;
    const float4* sphr;       // 16 B per REFERENCE (same order as refs): bounding sphere of the referenced triangle (see cull_sphere)
    const double* shd;
};

struct DevObject {
    int geom;       // rm::GeometryKind
    int mat;        // rm_material_kind
    int grid;       // index into DevScene::grid
    int pad;
    double g[6];    // sphere: origin xyz, radius | plane: origin xyz, normal xyz
    double color[3];// colour (Diffuse/Metal) or emitted radiance
    double rough;
};

struct DevScene {
    int n_objects;
    int n_grids;
    DevObject obj[kMaxObjects];
    DevGrid grid[kMaxGrids];
};

struct DevCamera {
    double pos[3];
    double width, height, aspect, tan_half;   // tan(fov_vert / 2 * PI / 180), evaluated once on the host (glibc)
    double focal_length, aperture_radius;
    int W, H;
    int use_dof;
    int pad;
};

// Ray queue of one stage, SoA: ray (6), throughput (3), path slot.
struct Queue {
    double* f[9];
    unsigned* id;
};

// Closest hit so far per ray of the current stage.
struct HitArrays {
    double* t;
    int* obj;        // -1 = miss
    unsigned* sub;
};

// Traversal queue: one 128-byte record per (ray, grid) pair that passed the AABB test:
//   [o.xyz d.x] [d.yz tmax.xy] [tmax.z tdelta.xyz] [cell.x cell.y | cell.z stepbits | ray index, - | -]
constexpr int kTravDoubles = 16;

struct DevTotals {
    unsigned long long samples, rays, nonfinite;
    unsigned long long stage_rays[RM_STAGE_SLOTS], grid_rays[RM_STAGE_SLOTS], cells[RM_STAGE_SLOTS], tests[RM_STAGE_SLOTS], shaded[RM_STAGE_SLOTS], survivors[RM_STAGE_SLOTS], occupied[RM_STAGE_SLOTS], test_flops[RM_STAGE_SLOTS];
};

// Per-batch device counters, all indexed by depth (zeroed once per batch).
struct StageCounters {
    unsigned* rays;       // rays[d]     = rays queued for depth d+1 (written by k_shade of depth d)
    unsigned* trav;       // trav[d]     = traversal records of depth d
    unsigned* cursor;     // cursor[d]   = fetch cursor of k_traverse at depth d
};

struct RenderParams {
    DevCamera cam;
    unsigned long long seed;
    const unsigned* pixel_map;   // owned pixel q -> frame pixel index (y*W + x), warp = 8x4 block
    unsigned n_pixels;           // owned pixels
    unsigned first_sample, sample_stride;
    unsigned bounce_limit;
    unsigned cap;                // paths per batch (capacity of queues and of `contrib`)
    double* contrib;             // 3 planes of `cap`: radiance each path delivered
    StageCounters cnt;
    DevTotals* totals;
};

__host__ __device__ inline unsigned stage_slot(unsigned depth) { return depth < RM_STAGE_SLOTS - 1 ? depth : RM_STAGE_SLOTS - 1; }

// ===================================================================== device math (cgmath semantics)

struct D3 { double x, y, z; };
__device__ __forceinline__ D3 d3(double x, double y, double z) { D3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ D3 operator+(D3 a, D3 b) { return d3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ D3 operator-(D3 a, D3 b) { return d3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ D3 operator-(D3 a) { return d3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ D3 operator*(D3 a, double s) { return d3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ D3 operator*(double s, D3 a) { return d3(s * a.x, s * a.y, s * a.z); }
// a / b for the shading weights, where a is very often exactly zero (black walls, a Smith term clamped to zero): CUDA's
// f64 division leaves its inline fast path for a zero dividend and calls a ~70-instruction subroutine, which showed up as
// 30 % of k_shade's instructions at 5 active lanes.  IEEE: (+-0) / b = +-0 with the XOR of the signs for every b that is
// neither zero nor NaN, so that case is answered directly; everything else is the ordinary division.
__device__ __forceinline__ double div0(double a, double b) {
    if (a == 0.0 && b == b && b != 0.0)
        return __longlong_as_double((__double_as_longlong(a) ^ __double_as_longlong(b)) & (long long)0x8000000000000000ull);
    return a / b;
}
__device__ __forceinline__ D3 operator/(D3 a, double s) { return d3(div0(a.x, s), div0(a.y, s), div0(a.z, s)); }
__device__ __forceinline__ D3 mul(D3 a, D3 b) { return d3(a.x * b.x, a.y * b.y, a.z * b.z); }
// Vector3::dot: products summed left to right
__device__ __forceinline__ double dot(D3 a, D3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
__device__ __forceinline__ D3 cross(D3 a, D3 b) { return d3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
// InnerSpace::normalize: multiply by the reciprocal magnitude
__device__ __forceinline__ D3 normalize(D3 a) { return a * (1.0 / sqrt(dot(a, a))); }
__device__ __forceinline__ double dist(D3 a, D3 b) { D3 d = b - a; return sqrt(dot(d, d)); }
// Matrix3::from_cols(c0, c1, c2) * v
__device__ __forceinline__ D3 mat_mul(D3 c0, D3 c1, D3 c2, D3 v) { return (c0 * v.x + c1 * v.y) + c2 * v.z; }
__device__ __forceinline__ D3 ld3(const double* p) { return d3(p[0], p[1], p[2]); }

// 256-bit global accesses (LDG/STG.E.ENL2.256 on sm_100a)
__device__ __forceinline__ void ld256_nc(const double* p, double& a, double& b, double& c, double& d) {
    asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void ld256(const double* p, double& a, double& b, double& c, double& d) {
    asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ void st256(double* p, double a, double b, double c, double d) {
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

// ===================================================================== intersection (bit-exact scope)

// Sphere::intersects                                       primitives/sphere.rs:11-27
__device__ __forceinline__ bool hit_sphere(const DevObject& s, D3 o, D3 d, double& t_out) {
    D3 c = ld3(s.g) - o;
    double t = dot(c, d);
    D3 q = c - t * d;
    double p = dot(q, q);
    double r2 = s.g[3] * s.g[3];
    if (p > r2) return false;
    t -= sqrt(r2 - p);
    if (t <= 0.0) return false;
    t_out = t;
    return true;
}

// Plane::intersects                                        primitives/plane.rs:11-24
__device__ __forceinline__ bool hit_plane(D3 origin, D3 normal, D3 o, D3 d, double& t_out) {
    double denom = dot(normal, -d);
    if (denom > 1e-6) {
        D3 p0l0 = origin - o;
        double t = dot(p0l0, -normal) / denom;
        if (t >= 0.0) { t_out = t; return true; }
    }
    return false;
}

// cgmath cast::<i32>(): Some(trunc) iff i32::MIN - 1 < v < i32::MAX + 1 (NaN fails)
__device__ __forceinline__ bool cast_i32(double v, int& out) {
    if (!(v > -2147483649.0 && v < 2147483648.0)) return false;
    out = __double2int_rz(v);
    return true;
}

// State of one ray inside AccGrid::intersects' loop (acc_grid.rs:127-184).
struct Dda {
    double tmx, tmy, tmz;   // t_max_{x,y,z}
    double tdx, tdy, tdz;   // t_delta_{x,y,z}
    int cx, cy, cz;         // current_cell
    unsigned step;          // bit a set: step along axis a is -1 (else +1)
};

// AABB::intersects (aabb.rs:10-31) followed by the set-up half of AccGrid::intersects
// (acc_grid.rs:90-125).  Returns false when the reference returns None before its loop (or would
// panic on a failed cast).  `tmin_out` / `tmax_out` are the AABB entry (may be negative) and exit distances.
// Quirks kept: only a NEGATIVE start cell is moved to the box entry point (A3); casts truncate
// toward zero (A5); signum looks at the sign bit, so -0.0 steps backwards (A7).
__device__ __forceinline__ bool grid_enter(const DevGrid& g, D3 o, D3 d, Dda& s, double& tmin_out, double& tmax_out) {
    const double ix = 1.0 / d.x, iy = 1.0 / d.y, iz = 1.0 / d.z;
    double t1 = (g.bmin[0] - o.x) * ix, t2 = (g.bmax[0] - o.x) * ix;
    double tmin = fmin(t1, t2), tmax = fmax(t1, t2);
    t1 = (g.bmin[1] - o.y) * iy; t2 = (g.bmax[1] - o.y) * iy;
    tmin = fmax(tmin, fmin(t1, t2)); tmax = fmin(tmax, fmax(t1, t2));
    t1 = (g.bmin[2] - o.z) * iz; t2 = (g.bmax[2] - o.z) * iz;
    tmin = fmax(tmin, fmin(t1, t2)); tmax = fmin(tmax, fmax(t1, t2));
    if (!(tmax > fmax(tmin, 0.0))) return false;
    tmin_out = tmin;
    tmax_out = tmax;

    const double csx = g.cell[0], csy = g.cell[1], csz = g.cell[2];
    double sx = o.x - g.bmin[0], sy = o.y - g.bmin[1], sz = o.z - g.bmin[2];
    int cx, cy, cz;
    if (!cast_i32(sx / csx, cx) || !cast_i32(sy / csy, cy) || !cast_i32(sz / csz, cz)) return false;
    if (cx < 0 || cy < 0 || cz < 0) {
        sx = (o.x + d.x * tmin) - g.bmin[0];   // outer_hit_position - bounding_box.min
        sy = (o.y + d.y * tmin) - g.bmin[1];
        sz = (o.z + d.z * tmin) - g.bmin[2];
        if (!cast_i32(sx / csx, cx) || !cast_i32(sy / csy, cy) || !cast_i32(sz / csz, cz)) return false;
    }
    if (d.x != d.x || d.y != d.y || d.z != d.z) return false;   // signum(NaN).cast() fails
    const bool nx = d.x < 0.0, ny = d.y < 0.0, nz = d.z < 0.0;
    s.step = (__double2hiint(d.x) < 0 ? 1u : 0u) | (__double2hiint(d.y) < 0 ? 2u : 0u) | (__double2hiint(d.z) < 0 ? 4u : 0u);
    s.tdx = (nx ? -csx : csx) / d.x;
    s.tdy = (ny ? -csy : csy) / d.y;
    s.tdz = (nz ? -csz : csz) / d.z;
    s.tmx = (((double)(cx + (nx ? 0 : 1)) * csx) - sx) / d.x;
    s.tmy = (((double)(cy + (ny ? 0 : 1)) * csy) - sy) / d.y;
    s.tmz = (((double)(cz + (nz ? 0 : 1)) * csz) - sz) / d.z;
    s.cx = cx; s.cy = cy; s.cz = cz;
    return true;
}

// Cell index with the reference's z stride of res.z (A1); false when it is >= cells.len()
// (acc_grid.rs:128-131: the traversal returns None).
__device__ __forceinline__ bool grid_cell_index(const DevGrid& g, int cx, int cy, int cz, unsigned long long& idx) {
    idx = (unsigned long long)(long long)cx +
          (unsigned long long)g.res[0] * ((unsigned long long)(long long)cy + (unsigned long long)(long long)cz * (unsigned long long)g.res[2]);
    return idx < g.n_cells;
}

// One step of the 3D-DDA (acc_grid.rs:155-183); ties go to the later axis (A4).  False = left the grid.
// Written with selects instead of the reference's four branches: the lanes of a warp step along different
// axes, and the arithmetic of the chosen axis (one compare pair, one integer add, one f64 add) is the same.
__device__ __forceinline__ bool dda_step(const DevGrid& g, Dda& s) {
    const bool xy = s.tmx < s.tmy, xz = s.tmx < s.tmz, yz = s.tmy < s.tmz;
    const bool ax = xy && xz;              // x
    const bool ay = !xy && yz;             // y; otherwise z
    const unsigned bit = ax ? 1u : (ay ? 2u : 4u);
    const int dir = (s.step & bit) ? -1 : 1;
    const int c = (ax ? s.cx : (ay ? s.cy : s.cz)) + dir;
    const int r = ax ? g.res[0] : (ay ? g.res[1] : g.res[2]);
    if (c >= r || c < 0) return false;
    const double tm = (ax ? s.tmx : (ay ? s.tmy : s.tmz)) + (ax ? s.tdx : (ay ? s.tdy : s.tdz));
    if (ax) { s.cx = c; s.tmx = tm; } else if (ay) { s.cy = c; s.tmy = tm; } else { s.cz = c; s.tmz = tm; }
    return true;
}

// The same step as predicated instructions (what the hot loop of k_traverse runs): three f64 compares choose the
// axis, then one integer add, one f64 add and one unsigned range check execute under that axis' predicate.
// sx/sy/sz = the reference's `step` (+1 / -1).  t_max of a ray that leaves the grid is advanced too; it is dead.
__device__ __forceinline__ bool dda_step_pred(double& tmx, double& tmy, double& tmz, double tdx, double tdy, double tdz, int& cx, int& cy, int& cz,
                                              int sx, int sy, int sz, unsigned rx, unsigned ry, unsigned rz) {
    unsigned alive;
    asm("{\n\t"
        ".reg .pred xy, xz, yz, px, py, pz, t, out;\n\t"
        "setp.lt.f64 xy, %0, %1;\n\t"
        "setp.lt.f64 xz, %0, %2;\n\t"
        "setp.lt.f64 yz, %1, %2;\n\t"
        "and.pred px, xy, xz;\n\t"
        "not.pred t, xy;\n\t"
        "and.pred py, t, yz;\n\t"
        "or.pred t, px, py;\n\t"
        "not.pred pz, t;\n\t"
        "@px add.s32 %3, %3, %10;\n\t"
        "@py add.s32 %4, %4, %11;\n\t"
        "@pz add.s32 %5, %5, %12;\n\t"
        "@px add.f64 %0, %0, %7;\n\t"
        "@py add.f64 %1, %1, %8;\n\t"
        "@pz add.f64 %2, %2, %9;\n\t"
        "setp.ge.and.u32 out, %3, %13, px;\n\t"
        "setp.ge.and.u32 t, %4, %14, py;\n\t"
        "or.pred out, out, t;\n\t"
        "setp.ge.and.u32 t, %5, %15, pz;\n\t"
        "or.pred out, out, t;\n\t"
        "selp.u32 %6, 0, 1, out;\n\t"
        "}"
        : "+d"(tmx), "+d"(tmy), "+d"(tmz), "+r"(cx), "+r"(cy), "+r"(cz), "=r"(alive)
        : "d"(tdx), "d"(tdy), "d"(tdz), "r"(sx), "r"(sy), "r"(sz), "r"(rx), "r"(ry), "r"(rz));
    return alive != 0u;
}

// Triangle::intersects (Moller-Trumbore, two-sided, eps 1e-8)     primitives/triangle.rs:11-44
struct TriPos { double v0x, v0y, v0z, v1x, v1y, v1z, v2x, v2y, v2z; };
__device__ __forceinline__ TriPos load_triangle(const double* __restrict__ tp) {
    TriPos p;
    double p0, p1, p2;
    ld256_nc(tp, p.v0x, p.v0y, p.v0z, p.v1x);
    ld256_nc(tp + 4, p.v1y, p.v1z, p.v2x, p.v2y);
    ld256_nc(tp + 8, p.v2z, p0, p1, p2);
    return p;
}
// `flops` (instrumented builds): the add / sub / mul / div count of the exit taken — 20, 30, 46 or 52 (SURVEY 8a, a20)
__device__ __forceinline__ bool hit_triangle(const TriPos& p, D3 o, D3 d, double& t_out, unsigned* flops = nullptr) {
    const D3 e1 = d3(p.v1x - p.v0x, p.v1y - p.v0y, p.v1z - p.v0z);
    const D3 e2 = d3(p.v2x - p.v0x, p.v2y - p.v0y, p.v2z - p.v0z);
    const D3 h = cross(d, e2);
    const double a = dot(e1, h);
    if (flops) *flops = 20u;
    if (a < 0.00000001 && a > -0.00000001) return false;
    const double f = 1.0 / a;
    const D3 s = d3(o.x - p.v0x, o.y - p.v0y, o.z - p.v0z);
    const double u = f * dot(s, h);
    if (flops) *flops = 30u;
    if (u < 0.0 || u > 1.0) return false;
    const D3 q = cross(s, e1);
    const double v = f * dot(d, q);
    if (flops) *flops = 46u;
    if (v < 0.0 || u + v > 1.0) return false;
    const double t = f * dot(e2, q);
    if (flops) *flops = 52u;
    if (!(t > 0.00000001)) return false;
    t_out = t;
    return true;
}

// Conservative pre-test of Triangle::intersects: true = the (infinite) line of the ray stays outside the triangle's bounding
// sphere by so much that the reference's f64 Moller-Trumbore arithmetic is certain to return None, so the candidate can be
// dropped without evaluating it.  The record holds an f32 centre c and an f32 radius R >= r (1 + 1e-6) + 1e-9 (1 + |c|) +
// |c - c_exact| (rounded up), r = distance from the exact centre to the farthest vertex.  All arithmetic here is f64:
// |cross(c - o, d)|^2 > R^2 |d|^2  <=>  distance(line, c) > R.  Rounding of the cross product is <= ~9e-16 |c - o| |d|,
// covered by the 1e-6 relative inflation whenever |c - o|^2 < 1e17 R^2; `lim` = 1.01e-17 * (largest squared distance
// from the ray origin to the grid's box, which holds every centre) is that guard, evaluated once per ray (else: not
// culled).  The reference's own rounding can move its barycentrics by <= ~1e-9 of an edge, orders of magnitude inside
// the inflation.  NaN compares false: not culled.
__device__ __forceinline__ bool cull_sphere(float4 sp, D3 o, D3 d, double dd, double lim) {
    const double r2 = (double)sp.w * (double)sp.w;
    const D3 oc = d3((double)sp.x - o.x, (double)sp.y - o.y, (double)sp.z - o.z);
    const D3 cr = cross(oc, d);
    return dot(cr, cr) > r2 * dd && lim < r2;
}

// Scene::intersect keeps the first object among equal distances (strict <, scene.rs:61).  Objects are
// not visited in index order here (analytic ones first, grids after), so the same rule is applied in
// its order-independent form: smaller distance wins, equal distances go to the lower object index.
__device__ __forceinline__ bool closer(double t, int obj, double best_t, int best_obj) {
    return best_obj < 0 || t < best_t || (t == best_t && obj < best_obj);
}

// ===================================================================== counter-based RNG
// Philox4x32-10, key = seed, counter = (pixel, sample, depth, draw >> 1).  Draw `i` of
// (pixel, sample, depth) stands in for the i-th rand::random::<f64>() the reference makes there.

__device__ __forceinline__ void philox(unsigned long long seed, unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned w[4]) {
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const unsigned h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const unsigned h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    w[0] = c0; w[1] = c1; w[2] = c2; w[3] = c3;
}
// 52 bits -> (k + 0.5) * 2^-52, strictly inside (0, 1)
__device__ __forceinline__ double u52(unsigned hi, unsigned lo) {
    const unsigned long long bits = ((unsigned long long)hi << 32) | lo;
    return (__ull2double_rn(bits >> 12) + 0.5) * (1.0 / 4503599627370496.0);
}

// ===================================================================== camera

// generate_primary_ray                                     src/trace.rs:322-333
// jx, jy are the jitter terms (rand - 0.5).
__device__ __forceinline__ D3 primary_direction(const DevCamera& c, unsigned xi, unsigned yi, double jx, double jy) {
    const double x = (double)xi + jx;
    const double y = (double)yi + jy;
    const double px = (2.0 * ((x + 0.5) / c.width) - 1.0) * c.tan_half * c.aspect;
    const double py = (1.0 - 2.0 * ((y + 0.5) / c.height)) * c.tan_half;
    return normalize(d3(px, py, 1.0));
}

// generate_primary_ray / generate_primary_ray_with_dof     src/trace.rs:322-360
__device__ __forceinline__ void camera_ray(const DevCamera& c, unsigned long long seed, unsigned pixel, unsigned sample, D3& o, D3& d) {
    unsigned w[4];
    philox(seed, pixel, sample, 0u, 0u, w);
    const unsigned xi = pixel % (unsigned)c.W, yi = pixel / (unsigned)c.W;
    const D3 cam = ld3(c.pos);
    D3 dir = primary_direction(c, xi, yi, u52(w[0], w[1]) - 0.5, u52(w[2], w[3]) - 0.5);
    if (!c.use_dof) { o = cam; d = dir; return; }
    // rejection-sample the aperture disk (world XY at the camera's z)
    D3 start;
    for (unsigned j = 1;; j++) {
        philox(seed, pixel, sample, 0u, j, w);
        const double r1 = u52(w[0], w[1]) * 2.0 - 1.0;
        const double r2 = u52(w[2], w[3]) * 2.0 - 1.0;
        start = d3(cam.x + r1 * c.aperture_radius, cam.y + r2 * c.aperture_radius, cam.z);
        if (dist(start, cam) < c.aperture_radius) break;
    }
    // focal plane: origin = cam + (0,0,1)*focal_length, normal (0,0,-1); Plane::intersects(primary).unwrap()
    const D3 fo = cam + d3(0.0, 0.0, 1.0) * c.focal_length;
    double t = 0.0;
    hit_plane(fo, d3(0.0, 0.0, -1.0), cam, dir, t);
    const D3 end = cam + t * dir;
    o = start;
    d = normalize(end - start);
}

// ===================================================================== shading (statistical scope)

// create_coordinate_system_of_n                            src/trace.rs:408-416
__device__ __forceinline__ void onb(D3 n, D3& t, D3& b) {
    const double sign = n.z > 0.0 ? 1.0 : -1.0;
    const double a = -1.0 / (sign + n.z);
    const double bb = n.x * n.y * a;
    t = d3(1.0 + sign * n.x * n.x * a, sign * bb, -sign * n.x);
    b = d3(bb, sign + n.y * n.y * a, -n.y);
}

__device__ __forceinline__ double pow5(double x) { const double x2 = x * x; return x2 * x2 * x; }

// Triangle::get_surface_properties (Heron-area barycentrics)    triangle.rs:47-68
__device__ __forceinline__ double heron(D3 a, D3 b, D3 c) {
    const double ab = dist(a, b), ac = dist(a, c), bc = dist(b, c);
    const double s = (ab + ac + bc) / 2.0;
    return sqrt(s * (s - ab) * (s - ac) * (s - bc));
}
__device__ __forceinline__ D3 triangle_normal(const DevGrid& g, unsigned ti, D3 p) {
    const double* tp = g.shd + (size_t)ti * 18;
    const D3 v0 = ld3(tp), v1 = ld3(tp + 3), v2 = ld3(tp + 6);
    const D3 n0 = ld3(tp + 9), n1 = ld3(tp + 12), n2 = ld3(tp + 15);
    const double abc = heron(v0, v1, v2);
    const double abp = heron(v0, v1, p);
    const double bcp = heron(v0, v2, p);
    const double ba = abp / abc, bb = bcp / abc;
    const double bc = 1.0 - (ba + bb);
    return normalize((n2 * ba) + (n1 * bb) + (n0 * bc));
}

// ---- f32 helpers of the statistical scope (RM_PRECISION_F32_SHADING).  The TU is compiled with -fmad=false (the bit-exact
// scope must not contract), so the FMAs here are written out.
struct F3 { float x, y, z; };
__device__ __forceinline__ F3 f3(float x, float y, float z) { F3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ F3 f3(D3 a) { return f3((float)a.x, (float)a.y, (float)a.z); }
__device__ __forceinline__ F3 operator+(F3 a, F3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ F3 operator*(F3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float dotf(F3 a, F3 b) { return fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)); }
__device__ __forceinline__ F3 normalizef(F3 a) { return a * rsqrtf(dotf(a, a)); }
// a * s + b
__device__ __forceinline__ F3 madf(F3 a, float s, F3 b) { return f3(fmaf(a.x, s, b.x), fmaf(a.y, s, b.y), fmaf(a.z, s, b.z)); }
__device__ __forceinline__ float pow5f(float x) { const float x2 = x * x; return x2 * x2 * x; }
// 23 bits -> (k + 0.5) * 2^-23: exactly representable, strictly inside (0, 1)
__device__ __forceinline__ float u23(unsigned w) { return ((float)(w >> 9) + 0.5f) * (1.0f / 8388608.0f); }
// sin / cos of an angle of any size the GGX lobe produces (theta = a sqrt(r / (1 - r)) <= ~4100 a with 23-bit uniforms): two-term
// Cody-Waite reduction to [-pi, pi], then the hardware approximations (abs. error ~5e-7, far below the Monte-Carlo noise)
__device__ __forceinline__ void sincos_reduced(float x, float& s, float& c) {
    const float k = rintf(x * 0.15915494309189535f);
    float r = fmaf(-k, 6.2831854820251465f, x);
    r = fmaf(-k, -1.7484555314695172e-07f, r);
    s = __sinf(r);
    c = __cosf(r);
}

// The lobe choice, direction sample and BRDF weight of one bounce (src/trace.rs:256-319) in f64 exactly as written: the
// reference's operations in the reference's order.  normal / view are unit vectors; returns the next direction, the weight the
// child radiance is multiplied by, and the ray offset along the normal.
__device__ __forceinline__ void lobe_f64(const RenderParams& rp, D3 normal, D3 to_camera, D3 color, double rough, double metal, unsigned pixel, unsigned sample,
                                         unsigned depth, D3& dir_out, D3& wgt, double& eps) {
    const D3 view = normalize(to_camera);                                   // :256 (always towards the camera position)
    const D3 f0 = d3(0.04 + metal * (color.x - 0.04), 0.04 + metal * (color.y - 0.04), 0.04 + metal * (color.z - 0.04));
    unsigned w[4];
    philox(rp.seed, pixel, sample, depth, 0u, w);
    const double r = u52(w[0], w[1]);                                       // :260
    const double ra = u52(w[2], w[3]);
    philox(rp.seed, pixel, sample, depth, 1u, w);
    const double rb = u52(w[0], w[1]);
    const double prob_d = 0.5 + metal * (0.0 - 0.5);                        // :263
    // The two lobes of :264-319 share most of their arithmetic (frame around an axis, normalisations, half vector,
    // one sincos), so only what differs is branched: a warp holds both kinds of sample.  Per path the operations
    // and their order are the reference's.
    const bool diffuse_lobe = r < prob_d;
    const double kTwoPi = 2.0 * 3.14159265358979323846;
    D3 axis;
    double s_t, c_t, phi;            // sin / cos of the polar angle, azimuth
    if (diffuse_lobe) {
        // cosine-weighted hemisphere: theta = acos(sqrt(r1)), pdf = sqrt(r1)      :396-406
        c_t = sqrt(ra); s_t = sqrt(1.0 - ra);
        phi = kTwoPi * rb;
        axis = normal;
        eps = 0.00001;                                                          // :269
    } else {
        axis = normalize(-view - 2.0 * (-dot(view, normal) * normal));          // reflect :285
        const double a = rough * rough;
        phi = kTwoPi * ra;
        const double theta = a * sqrt(rb / (1.0 - rb));                         // :291 (used as an angle)
        sincos(theta, &s_t, &c_t);
        eps = 0.0001;                                                           // :300
    }
    double sp, cp;
    sincos(phi, &sp, &cp);
    D3 tg, bt;
    onb(axis, tg, bt);
    const D3 dir = normalize(mat_mul(tg, axis, bt, d3(s_t * cp, c_t, s_t * sp)));   // :266 / :295
    const double ndl = dot(normal, dir);                                        // :275 / :306
    const D3 light = diffuse_lobe ? dir : normalize(dir);                       // :307 (the specular lobe normalises again)
    const D3 half = normalize(light + view);                                    // :276 / :308
    const double hv = dot(half, view);
    const D3 one = d3(1.0, 1.0, 1.0);
    if (diffuse_lobe) {
        const double cos_theta = fmax(ndl, 0.0);                                // :275
        const D3 fres = f0 + (one - f0) * pow5(1.0 - fmax(hv, 0.0));            // :277
        const D3 diff = (one - fres) * (1.0 - metal);
        wgt = (mul(diff, color) * cos_theta) / (prob_d * c_t);                  // :281-282
    } else {
        const D3 F = f0 + (one - f0) * pow5(1.0 - hv);                          // :309
        const double a2 = rough * rough;                                        // ggx_distribution :362-370
        const double nh = dot(normal, half);
        double den = (nh * nh) * (a2 - 1.0) + 1.0;
        den = fmax(3.14159265358979323846 * den * den, 1e-7);
        const double D = a2 / den;
        const double k = (rough * rough) / 8.0;                                 // geometry_smith :372-382
        const double nv = fmax(dot(normal, view), 0.0), nl = fmax(ndl, 0.0);
        const double G = div0(nv, nv * (1.0 - k) + k) * div0(nl, nl * (1.0 - k) + k);
        const D3 nom = (D * G) * F;
        const double denom = 4.0 * dot(normal, view) * ndl + 0.001;             // :313
        const double pdf = (D * nh) / (4.0 * hv) + 0.0001;                      // :317
        wgt = (((nom / denom) * ndl) / (1.0 - prob_d)) / pdf;
    }
    dir_out = dir;
}

// The same bounce with the statistical scope in f32 (RM_PRECISION_F32_SHADING): same formulas, same lobe probabilities, 23-bit
// uniforms from one Philox call, FMAs, rsqrt normalisations.  The result agrees with lobe_f64 to ~1e-6 relative, i.e. far
// inside the Monte-Carlo noise the image tolerance of SURVEY 8d is defined by; the direction is re-normalised in f64 so the
// intersection code downstream still sees |d| = 1 to f64 accuracy.
__device__ __forceinline__ void lobe_f32(const RenderParams& rp, D3 normal64, D3 to_camera, D3 color64, double rough64, double metal64, unsigned pixel,
                                         unsigned sample, unsigned depth, D3& dir_out, D3& wgt_out, double& eps) {
    const F3 normal = f3(normal64), view = normalizef(f3(to_camera)), color = f3(color64);
    const float rough = (float)rough64, metal = (float)metal64;
    const F3 f0 = f3(fmaf(metal, color.x - 0.04f, 0.04f), fmaf(metal, color.y - 0.04f, 0.04f), fmaf(metal, color.z - 0.04f, 0.04f));
    unsigned w[4];
    philox(rp.seed, pixel, sample, depth, 0u, w);
    const float r = u23(w[0]), ra = u23(w[2]), rb = u23(w[1]);
    const float prob_d = 0.5f - 0.5f * metal;
    const bool diffuse_lobe = r < prob_d;
    F3 axis;
    float s_t, c_t, sp, cp;
    if (diffuse_lobe) {
        c_t = sqrtf(ra); s_t = sqrtf(1.0f - ra);
        sincospif(2.0f * rb, &sp, &cp);
        axis = normal;
        eps = 0.00001;
    } else {
        axis = normalizef(madf(normal, 2.0f * dotf(view, normal), f3(-view.x, -view.y, -view.z)));
        sincospif(2.0f * ra, &sp, &cp);
        sincos_reduced((rough * rough) * sqrtf(__fdividef(rb, 1.0f - rb)), s_t, c_t);
        eps = 0.0001;
    }
    // create_coordinate_system_of_n (:408-416) around the axis, then Matrix3::from_cols(t, axis, b) * (s cos, c, s sin)
    const float sign = axis.z > 0.0f ? 1.0f : -1.0f;
    const float a_ = -1.0f / (sign + axis.z);
    const float bb = axis.x * axis.y * a_;
    const F3 tg = f3(fmaf(sign * axis.x, axis.x * a_, 1.0f), sign * bb, -sign * axis.x);
    const F3 bt = f3(bb, fmaf(axis.y, axis.y * a_, sign), -axis.y);
    const F3 dir = normalizef(madf(bt, s_t * sp, madf(axis, c_t, tg * (s_t * cp))));
    const float ndl = dotf(normal, dir);
    const F3 half = normalizef(dir + view);
    const float hv = dotf(half, view);
    F3 wgt;
    if (diffuse_lobe) {
        const float cos_theta = fmaxf(ndl, 0.0f);
        const float fr = pow5f(1.0f - fmaxf(hv, 0.0f));
        const float scale = (1.0f - metal) * cos_theta / (prob_d * c_t);
        wgt = f3((1.0f - fmaf(1.0f - f0.x, fr, f0.x)) * color.x * scale, (1.0f - fmaf(1.0f - f0.y, fr, f0.y)) * color.y * scale,
                 (1.0f - fmaf(1.0f - f0.z, fr, f0.z)) * color.z * scale);
    } else {
        const float fr = pow5f(1.0f - hv);
        const float a2 = rough * rough;
        const float nh = dotf(normal, half);
        float den = fmaf(nh * nh, a2 - 1.0f, 1.0f);
        den = fmaxf(3.14159265358979323846f * den * den, 1e-7f);
        const float D = a2 / den;
        const float k = a2 * 0.125f;
        const float nvs = dotf(normal, view);
        const float nv = fmaxf(nvs, 0.0f), nl = fmaxf(ndl, 0.0f);
        const float G = (nv / fmaf(nv, 1.0f - k, k)) * (nl / fmaf(nl, 1.0f - k, k));
        const float denom = fmaf(4.0f * nvs, ndl, 0.001f);
        const float pdf = fmaf(D * nh, 1.0f / (4.0f * hv), 0.0001f);
        const float scale = (D * G) / denom * ndl / (1.0f - prob_d) / pdf;
        wgt = f3(fmaf(1.0f - f0.x, fr, f0.x) * scale, fmaf(1.0f - f0.y, fr, f0.y) * scale, fmaf(1.0f - f0.z, fr, f0.z) * scale);
    }
    // |dir| = 1 to f32 accuracy; one Newton step of 1 / sqrt(|dir|^2) around 1 brings it to ~1e-14 without an f64 sqrt / division
    const D3 dd = d3((double)dir.x, (double)dir.y, (double)dir.z);
    dir_out = dd * (1.5 - 0.5 * dot(dd, dd));
    wgt_out = d3((double)wgt.x, (double)wgt.y, (double)wgt.z);
}

// One bounce of `trace` (src/trace.rs:232-320) in throughput form: the recursion multiplies the
// child radiance by a weight known before recursing, so a path's value is (prod of weights) (*)
// emission.  Returns true when the path continues with (o, d, T) updated; otherwise `result` is
// the radiance the path delivers.  PREC = rm_precision: the hit point, the surface normal and the next
// origin are f64 in both modes; the lobe sampling and the BRDF weight follow PREC.
// What one bounce does to a path, before the path's throughput T is involved (T is read from the queue only afterwards, so
// its six registers are free during the bounce): BOUNCE_NONE = the path ends with no radiance, BOUNCE_EMIT = it delivers
// T (*) v, BOUNCE_CONTINUE = it goes on from (o, d) with T (*) v.
// KEEP (RM_FLAG_KEEP_NONFINITE): at the bounce limit the last weight is still computed and returned in v with BOUNCE_NONE,
// because the reference multiplies the child's zero by it (:235-237, :281-282, :315-319) and a NaN / Inf weight makes the
// sample NaN.  The lobe's draws are counter-based, so the extra evaluation leaves every other draw unchanged.
enum Bounce : int { BOUNCE_NONE = 0, BOUNCE_EMIT = 1, BOUNCE_CONTINUE = 2 };

template <int PREC, bool KEEP>
__device__ __forceinline__ Bounce shade(const DevScene& sc, const RenderParams& rp, double hit_t, int hit_obj, unsigned hit_sub, unsigned pixel,
                                        unsigned sample, unsigned depth, D3& o, D3& d, D3& v, unsigned& shaded_tri) {
    if (hit_obj < 0) return BOUNCE_NONE;                                    // :242
    const DevObject& ob = sc.obj[hit_obj];
    const D3 frag = o + d * hit_t;                                          // :246
    if (ob.mat == RM_MATERIAL_EMISSION) { v = ld3(ob.color); return BOUNCE_EMIT; }   // :250
    if (!KEEP && depth >= rp.bounce_limit) return BOUNCE_NONE;              // the child call returns 0 (:235-237)
    D3 normal;                                                              // :244
    if (ob.geom == GEOM_PLANE) normal = ld3(ob.g + 3);
    else if (ob.geom == GEOM_SPHERE) normal = normalize(frag - ld3(ob.g));
    else { normal = triangle_normal(sc.grid[ob.grid], hit_sub, frag); shaded_tri++; }
    const D3 to_camera = ld3(rp.cam.pos) - frag;
    const double metal = ob.mat == RM_MATERIAL_METAL ? 1.0 : 0.0;
    D3 dir;
    double eps;
    if (PREC == RM_PRECISION_F32_SHADING) lobe_f32(rp, normal, to_camera, ld3(ob.color), ob.rough, metal, pixel, sample, depth, dir, v, eps);
    else lobe_f64(rp, normal, to_camera, ld3(ob.color), ob.rough, metal, pixel, sample, depth, dir, v, eps);
    if (KEEP && depth >= rp.bounce_limit) return BOUNCE_NONE;
    o = frag + normal * eps;
    d = dir;
    return BOUNCE_CONTINUE;
}

// ===================================================================== kernels

enum RaySource : int { SRC_CAMERA = 0, SRC_QUEUE = 1, SRC_AOS = 2 };

struct SetupArgs {
    const double* q[6];        // SRC_QUEUE: ray SoA of this stage;  SRC_CAMERA: the same arrays, written here
    const rm_ray* aos;         // SRC_AOS: caller's rays
    const unsigned* n_ptr;     // number of rays (device) ...
    unsigned n_direct;         // ... or, when n_ptr is null, this
    HitArrays hit;
    double* trav;              // traversal queue (kTravDoubles per record)
    unsigned* trav_count;
    int grid_object;           // object index of the grid this pass sets up, -1 = none
    int analytic;              // 1: evaluate the Sphere/Plane objects and initialise the hit record
    int emitters_only;         // 1: the grid can only matter when the closest hit so far is an emitter (see k_setup)
};

// Stage part 1.  See the header comment.
template <int SRC>
__global__ void __launch_bounds__(kBlock, RM_SETUP_BLOCKS_PER_SM) k_setup(const __grid_constant__ DevScene sc, const __grid_constant__ RenderParams rp,
                                                   const __grid_constant__ SetupArgs a) {
    const unsigned n = a.n_ptr ? *a.n_ptr : a.n_direct;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned warps_total = (gridDim.x * blockDim.x) >> 5;
    const unsigned warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    for (unsigned base = warp * 32u; base < n; base += warps_total * 32u) {
        const unsigned i = base + lane;
        bool push = false;
        D3 o, d;
        Dda s;
        double best_t = 0.0;        // closest hit among the objects already evaluated: travels with the traversal record
        int best_obj = -1;
        if (i < n) {
            if (SRC == SRC_CAMERA) {
                const unsigned q = i % rp.n_pixels, s_local = i / rp.n_pixels;
                camera_ray(rp.cam, rp.seed, rp.pixel_map[q], rp.first_sample + s_local * rp.sample_stride, o, d);
                double* const* w = const_cast<double* const*>(a.q);
                w[0][i] = o.x; w[1][i] = o.y; w[2][i] = o.z; w[3][i] = d.x; w[4][i] = d.y; w[5][i] = d.z;
            } else if (SRC == SRC_QUEUE) {
                o = d3(a.q[0][i], a.q[1][i], a.q[2][i]);
                d = d3(a.q[3][i], a.q[4][i], a.q[5][i]);
            } else {
                const double* r = reinterpret_cast<const double*>(a.aos + i);
                o = d3(r[0], r[1], r[2]);
                d = d3(r[3], r[4], r[5]);
            }
            if (a.analytic) {
                // Scene::intersect over the Sphere / Plane objects, in order, strict <   scene.rs:54-68
                double closest = DBL_MAX;
                for (int k = 0; k < sc.n_objects; k++) {
                    const DevObject& ob = sc.obj[k];
                    double t;
                    bool got = false;
                    if (ob.geom == GEOM_PLANE) got = hit_plane(ld3(ob.g), ld3(ob.g + 3), o, d, t);
                    else if (ob.geom == GEOM_SPHERE) got = hit_sphere(ob, o, d, t);
                    if (got && t < closest) { closest = t; best_t = t; best_obj = k; }
                }
                a.hit.t[i] = best_t;
                a.hit.obj[i] = best_obj;
                a.hit.sub[i] = 0u;
            } else {
                best_obj = a.hit.obj[i];
                best_t = a.hit.t[i];
            }
            // emitters_only (drop mode at the bounce limit, no grid object emits): the path delivers its throughput times the
            // emission of the closest object if that is an emitter, else an exact 0 (shade()).  A non-emissive grid can only
            // hide an emitter, so when the closest hit so far is not one, every answer of the traversal delivers the same 0.
            const bool decided = a.emitters_only && (best_obj < 0 || sc.obj[best_obj].mat != RM_MATERIAL_EMISSION);
            if (a.grid_object >= 0 && !decided) {
                const DevGrid& g = sc.grid[sc.obj[a.grid_object].grid];
                double tmin, tmax;
                push = grid_enter(g, o, d, s, tmin, tmax);
                // Every triangle lies inside the box, so the true distance of any grid hit is >= the box
                // entry distance.  If another object is already hit before the entry point by more than the
                // worst-case error of a computed triangle distance, the grid cannot win the strict `<` of
                // Scene::intersect and its traversal is skipped.  Error bound of Moller-Trumbore's t = f * dot(e2, cross(s, e1)):
                // c * eps * |s| * |e|^2 / |a| with |a| >= 1e-8 (triangle.rs:21), c * eps <= 4e-15, |e|^2 <= diag2 and
                // |s| = |o - v0| <= max(tmin, 0) + diag (v0 is in the box; the box is entered at distance max(tmin, 0), |d| = 1)
                // =>  <= 4e-7 * (max(tmin, 0) + diag) * diag2; plus 1e-6 absolute for the rounding of tmin itself.
                if (push && best_obj >= 0 && tmin > best_t + (1e-6 + 4e-7 * (fmax(tmin, 0.0) + g.diag) * g.diag2)) push = false;
            }
        }
        const unsigned mask = __ballot_sync(0xffffffffu, push);
        if (mask) {
            unsigned pos = 0;
            if (lane == 0) pos = atomicAdd(a.trav_count, (unsigned)__popc(mask));
            pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(mask & ((1u << lane) - 1u));
            if (push) {
                double* rec = a.trav + (size_t)pos * kTravDoubles;
                st256(rec, o.x, o.y, o.z, d.x);
                st256(rec + 4, d.y, d.z, s.tmx, s.tmy);
                st256(rec + 8, s.tmz, s.tdx, s.tdy, s.tdz);
                st256(rec + 12, __hiloint2double(s.cy, s.cx), __hiloint2double((int)s.step, s.cz), __hiloint2double(best_obj, (int)i), best_t);
            }
        }
    }
}

struct TraverseArgs {
    const double* trav;
    const unsigned* n_ptr;
    unsigned* cursor;
    HitArrays hit;
    int grid_object;       // object index reported for hits
    unsigned depth;        // for the work counters
    DevTotals* totals;
};

// Stage part 2: AccGrid::intersects' loop (acc_grid.rs:127-184) for every queued ray.
// Quirks kept: the first cell holding any hit returns its closest hit without an in-cell check (A2);
// the per-cell closest starts at 5712515.0 (A6); leaving the grid or an out-of-range cell index is a miss.
//
// Persistent warps.  Every lane owns one ray's DDA state; the triangle tests are NOT tied to the lane
// that owns the ray.  One loop iteration is three warp-uniform phases:
//   A  lanes whose ray needs a cell walk the DDA (a bounded number of steps) to the next non-empty cell
//   B  the triangle lists of all cells found are pooled: the warp's 32 lanes take (ray, reference) pairs
//      from the pool round-robin, so every lane tests a triangle in every round, the reference and
//      triangle fetches of a round are independent loads, and a ray's whole cell is tested in ~one L2
//      round trip instead of one per triangle.  Per cell the winner is the smallest distance, ties to
//      the earliest list position (the reference's strict `<` while walking the list in order)
//   C  rays with a hit are finished (hit record merged), the others go back to A
// Idle lanes re-fill from the traversal queue in groups.
#ifndef RM_TRAV_BLOCK
#define RM_TRAV_BLOCK 256
#endif
constexpr int kTravBlock = RM_TRAV_BLOCK;          // threads per block of k_traverse
constexpr int kTravWarps = kTravBlock / 32;
#ifndef RM_TRAV_MAX_STEPS
#define RM_TRAV_MAX_STEPS 2
#endif
#ifndef RM_TRAV_REFILL_MIN
#define RM_TRAV_REFILL_MIN 8
#endif
// 4 blocks of 256 threads = 32 warps per SM at 64 registers.  Possible since the DDA state, the ray index and the per-cell best hit
// live in shared memory outside the phases that use them (RM_TRAV_PARK): 12 B of spills, one reload inside the pooled round.
// 3 blocks (76 registers, no spills) is 3 % slower on the L2-resident GoldDragon and 1.5 % faster on multi-million-triangle soups.
#ifndef RM_TRAV_BLOCKS_PER_SM
#define RM_TRAV_BLOCKS_PER_SM 4
#endif
#ifndef RM_TRAV_LOOK
#define RM_TRAV_LOOK 4
#endif
constexpr unsigned kLook = RM_TRAV_LOOK;                  // cells looked ahead per walk iteration
constexpr unsigned kTravMaxSteps = RM_TRAV_MAX_STEPS;     // walk iterations per phase A
constexpr unsigned kRefillMin = RM_TRAV_REFILL_MIN;       // idle lanes that trigger a re-fill while others still have work

// RM_TRAV_PARK (default on): the lane's DDA state lives in shared memory between walks, see TravWarpShared::dda_t
#ifndef RM_TRAV_PARK
#define RM_TRAV_PARK 1
#endif
#ifndef RM_TRAV_EXCL_SHARED
#define RM_TRAV_EXCL_SHARED 1
#endif
struct TravWarpShared {
    double2 ray[32][3];                // {o.x o.y} {o.z d.x} {d.y d.z} of the lane's ray (three 128-bit accesses)
    unsigned long long cand_t[32];     // this round's smallest distance bits per ray
    unsigned cand_tri[32];             // ... and the smallest triangle index that has it (= the earliest list position: a cell's list ascends)
    unsigned olane[32];                // q-th lane that contributes a list to the pool
    unsigned odelta[32];               // ... and (first reference of its cell) - (its first item): position = item + odelta
    double2 dd_lim[32];                // |d|^2 of the lane's ray, and the guard of cull_sphere
    unsigned s_tri[64];                // ring of candidates that survived the sphere pre-test: triangle index
    unsigned char s_owner[64];         // ... and the lane that owns the ray
    double best_t[32];                 // the lane's ray: closest hit among the objects evaluated before this grid (from the
    int best_obj[32];                  // traversal record), merged with the grid's answer when the ray finishes
#if RM_TRAV_PARK
    double dda_t[6][32];               // t_max xyz, t_delta xyz of the lane's ray while it is not walking (phase B / C): the DDA state
    int dda_c[3][32];                  // lives in registers only inside phase A, which lets the pooled loops run with 18 fewer
    unsigned dda_s[32];                // live registers (current cell; bit a set: step along axis a is -1)
    unsigned ray_index[32];            // index of the lane's ray in the stage's queue (needed once, when it finishes)
    unsigned long long cell_t[32];     // closest hit of the lane's ray in its current cell (distance bits, triangle): touched only
    unsigned cell_tri[32];             // when a round found a hit and when the ray finishes
    unsigned char state[32];           // the lane's TravState during the pooled phase
#endif
#if RM_TRAV_EXCL_SHARED
    unsigned excl[32];                 // first pool item of the lane's list (~0: none): read by locate() every round
#endif
};

enum TravState : unsigned { TS_IDLE = 0, TS_LOOK = 1, TS_STEP = 2, TS_READY = 3 };

#if defined(RM_TRAV_PROFILE)
// -DRM_TRAV_PROFILE: SM-clock cycles per phase, summed over warps (tuning builds only; read with rm_debug_trav_profile)
__device__ unsigned long long g_trav_prof[8];
#define RM_PROF_MARK(slot) do { const long long now__ = clock64(); prof[slot] += (unsigned long long)(now__ - prof_t); prof_t = now__; } while (0)
#else
#define RM_PROF_MARK(slot) do { } while (0)
#endif

template <bool COUNT>
__global__ void __launch_bounds__(kTravBlock, RM_TRAV_BLOCKS_PER_SM) k_traverse(const __grid_constant__ DevGrid g, const __grid_constant__ TraverseArgs a) {
    __shared__ TravWarpShared shared[kTravWarps];
    TravWarpShared& sh = shared[threadIdx.x >> 5];
    const unsigned n = *a.n_ptr;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt = (1u << lane) - 1u;
    const unsigned FULL = 0xffffffffu;
    constexpr unsigned long long kClosest0 = 0x4155CAA0C0000000ull;   // bits of 5712515.0 (acc_grid.rs:135)
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.totals) atomicAdd(&a.totals->grid_rays[stage_slot(a.depth)], (unsigned long long)n);

    unsigned state = TS_IDLE;
    bool exhausted = false;                 // the queue has no more records for this warp
    // DDA state of MY ray (acc_grid.rs:100-125)
#if !RM_TRAV_PARK
    double tmx = 0, tmy = 0, tmz = 0, tdx = 0, tdy = 0, tdz = 0;
    int cx = 0, cy = 0, cz = 0, sx = 1, sy = 1, sz = 1;
#endif
    const unsigned rx = (unsigned)g.res[0], ry = (unsigned)g.res[1], rz = (unsigned)g.res[2];
#if RM_TRAV_PARK
    unsigned k = 0, cnt = 0;
#else
    unsigned ray = 0, k = 0, cnt = 0;
#endif
    unsigned n_cells = 0, n_tests = 0, n_surv = 0, n_occ = 0, n_flops = 0;
#if defined(RM_TRAV_PROFILE)
    unsigned long long prof[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long prof_t = clock64();
#endif
    for (;;) {
        // ---- re-fill
        RM_PROF_MARK(4);
        const unsigned idle = __ballot_sync(FULL, state == TS_IDLE);
        if (idle == FULL && exhausted) break;
        if (!exhausted && (idle == FULL || __popc(idle) >= (int)kRefillMin)) {
            unsigned base = 0;
            if (lane == 0) base = atomicAdd(a.cursor, (unsigned)__popc(idle));
            base = __shfl_sync(FULL, base, 0);
            if (base + (unsigned)__popc(idle) >= n) exhausted = true;     // warp-uniform
            if (state == TS_IDLE) {
                const unsigned idx = base + __popc(idle & lt);
                if (idx < n) {
                    const double* rec = a.trav + (size_t)idx * kTravDoubles;
                    double ox, oy, oz, dx, dy, dz, q0, q1, q2, q3;
                    ld256(rec, ox, oy, oz, dx);
#if RM_TRAV_PARK
                    {
                        double t0, t1, t2, t3, t4, t5;
                        ld256(rec + 4, dy, dz, t0, t1);
                        ld256(rec + 8, t2, t3, t4, t5);
                        ld256(rec + 12, q0, q1, q2, q3);
                        sh.dda_t[0][lane] = t0; sh.dda_t[1][lane] = t1; sh.dda_t[2][lane] = t2;
                        sh.dda_t[3][lane] = t3; sh.dda_t[4][lane] = t4; sh.dda_t[5][lane] = t5;
                        sh.dda_c[0][lane] = __double2loint(q0); sh.dda_c[1][lane] = __double2hiint(q0); sh.dda_c[2][lane] = __double2loint(q1);
                        sh.dda_s[lane] = (unsigned)__double2hiint(q1);
                    }
#else
                    ld256(rec + 4, dy, dz, tmx, tmy);
                    ld256(rec + 8, tmz, tdx, tdy, tdz);
                    ld256(rec + 12, q0, q1, q2, q3);
                    cx = __double2loint(q0); cy = __double2hiint(q0); cz = __double2loint(q1);
                    const unsigned neg = (unsigned)__double2hiint(q1);
                    sx = (neg & 1u) ? -1 : 1; sy = (neg & 2u) ? -1 : 1; sz = (neg & 4u) ? -1 : 1;
#endif
#if RM_TRAV_PARK
                    sh.ray_index[lane] = (unsigned)__double2loint(q2);
#else
                    ray = (unsigned)__double2loint(q2);
#endif
                    sh.best_obj[lane] = __double2hiint(q2);
                    sh.best_t[lane] = q3;
                    sh.ray[lane][0] = make_double2(ox, oy);
                    sh.ray[lane][1] = make_double2(oz, dx);
                    sh.ray[lane][2] = make_double2(dy, dz);
                    {
                        const double mx = fmax(fabs(g.bmin[0] - ox), fabs(g.bmax[0] - ox)), my = fmax(fabs(g.bmin[1] - oy), fabs(g.bmax[1] - oy)),
                                     mz = fmax(fabs(g.bmin[2] - oz), fabs(g.bmax[2] - oz));
                        sh.dd_lim[lane] = make_double2((dx * dx + dy * dy) + dz * dz, ((mx * mx + my * my) + mz * mz) * 1.01e-17);
                    }
                    state = TS_LOOK;
                }
            }
        }
        RM_PROF_MARK(0);
        // ---- A: walk to the next non-empty cell.  The walk is a chain of dependent round trips (step -> occupancy word),
        // so each iteration looks kLook cells ahead: the DDA is advanced kLook times in registers (the arithmetic is
        // cheap and exactly the reference's sequence), the kLook occupancy words are fetched together, and the ray
        // commits up to the first occupied cell (re-walking from the saved state) or all kLook empty ones.
#if RM_TRAV_PARK
        double tmx = 0, tmy = 0, tmz = 0, tdx = 0, tdy = 0, tdz = 0;
        int cx = 0, cy = 0, cz = 0, sx = 1, sy = 1, sz = 1;
        const bool walking = state == TS_LOOK || state == TS_STEP;
        if (walking) {
            tmx = sh.dda_t[0][lane]; tmy = sh.dda_t[1][lane]; tmz = sh.dda_t[2][lane];
            tdx = sh.dda_t[3][lane]; tdy = sh.dda_t[4][lane]; tdz = sh.dda_t[5][lane];
            cx = sh.dda_c[0][lane]; cy = sh.dda_c[1][lane]; cz = sh.dda_c[2][lane];
            const unsigned neg = sh.dda_s[lane];
            sx = (neg & 1u) ? -1 : 1; sy = (neg & 2u) ? -1 : 1; sz = (neg & 4u) ? -1 : 1;
        }
#endif
#pragma unroll 1
        for (unsigned it = 0; it < kTravMaxSteps; it++) {
            if (state == TS_LOOK) {                              // a fresh ray: its start cell, no step (acc_grid.rs:127-131)
                unsigned long long ci;
                state = TS_IDLE;                                 // index >= cells.len(): the reference returns None
                if (grid_cell_index(g, cx, cy, cz, ci)) {
                    state = TS_STEP;
                    if (COUNT) n_cells++;
                    if ((__ldg(&g.occ[ci >> 5]) >> (ci & 31u)) & 1u) { k = (unsigned)ci; state = TS_READY; }
                }
            } else if (state == TS_STEP) {
                const double a0 = tmx, a1 = tmy, a2 = tmz;
                const int b0 = cx, b1 = cy, b2 = cz;
                unsigned idx[kLook], word[kLook];
                unsigned ended = kLook;                          // first look-ahead step at which the traversal ends without a cell
#pragma unroll
                for (unsigned j = 0; j < kLook; j++) {
                    idx[j] = 0u; word[j] = 0u;
                    if (ended == kLook) {
                        unsigned long long ci;
                        if (dda_step_pred(tmx, tmy, tmz, tdx, tdy, tdz, cx, cy, cz, sx, sy, sz, rx, ry, rz) && grid_cell_index(g, cx, cy, cz, ci)) {
                            idx[j] = (unsigned)ci;
                            word[j] = __ldg(&g.occ[ci >> 5]);
                        } else {
                            ended = j;                           // left the grid, or index >= cells.len(): None
                        }
                    }
                }
                unsigned first = kLook;                          // first occupied cell among the ones reached
#pragma unroll
                for (unsigned j = kLook; j-- > 0;)
                    if (j < ended && ((word[j] >> (idx[j] & 31u)) & 1u)) first = j;
                if (first < kLook) {
                    // commit first + 1 steps: re-walk from the saved state (same operations, same results)
                    tmx = a0; tmy = a1; tmz = a2; cx = b0; cy = b1; cz = b2;
#pragma unroll
                    for (unsigned j = 0; j < kLook; j++)
                        if (j <= first) dda_step_pred(tmx, tmy, tmz, tdx, tdy, tdz, cx, cy, cz, sx, sy, sz, rx, ry, rz);
                    k = idx[0];
#pragma unroll
                    for (unsigned j = 1; j < kLook; j++) if (j == first) k = idx[j];
                    state = TS_READY;
                    if (COUNT) n_cells += first + 1u;
                } else {
                    if (COUNT) n_cells += ended;
                    if (ended < kLook) state = TS_IDLE;          // the reference returns None
                }
            }
            if (!__any_sync(FULL, state == TS_STEP)) break;
        }
#if RM_TRAV_PARK
        if (walking) {
            sh.dda_t[0][lane] = tmx; sh.dda_t[1][lane] = tmy; sh.dda_t[2][lane] = tmz;
            sh.dda_c[0][lane] = cx; sh.dda_c[1][lane] = cy; sh.dda_c[2][lane] = cz;
        }
#endif
        // the cell records of every ray that found an occupied cell, in one round trip (not one per walk iteration)
        if (state == TS_READY) {
            const uint2 cell = __ldg(&g.cells[k]);
            k = cell.x; cnt = cell.y;
            if (COUNT) { n_tests += cnt; n_occ++; }
        }
        RM_PROF_MARK(1);
        // ---- B: pooled triangle tests of every ready cell
        const unsigned mine = state == TS_READY ? cnt : 0u;
        unsigned incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(FULL, incl, o);
            if ((int)lane >= o) incl += v;
        }
        const unsigned total = __reduce_add_sync(FULL, mine);        // warp-uniform by construction (a uniform register, not one per lane)
        if (total == 0) continue;
#if RM_TRAV_PARK
        sh.state[lane] = (unsigned char)state;                       // not needed until phase C
#endif
        // The pool: items [excl, excl + mine) belong to this lane's cell.  Contributing lanes are compacted into
        // olane / odelta; a round of 32 consecutive items finds its owners with one ballot and one redux:
        //   first = contributors whose list starts at or before the round, bits = list starts inside the round
        // first item of MY list; ~0 for a lane that contributes none (neither "at or before the round" nor "inside it": the two
        // tests of locate() need no separate flag)
        {
            const unsigned excl = mine ? incl - mine : ~0u;
#if RM_TRAV_EXCL_SHARED
            sh.excl[lane] = excl;
#endif
            const unsigned contrib = __ballot_sync(FULL, mine != 0u);
            if (mine) {
                const unsigned q = __popc(contrib & lt);
                sh.olane[q] = lane;
                sh.odelta[q] = k - excl;
            }
        }
#if !RM_TRAV_EXCL_SHARED
        const unsigned excl = mine ? incl - mine : ~0u;
#endif
        sh.cand_t[lane] = ~0ull;
        sh.cand_tri[lane] = ~0u;
#if RM_TRAV_PARK
        sh.cell_t[lane] = kClosest0;                 // per-cell closest of MY ray
        sh.cell_tri[lane] = ~0u;
#else
        unsigned long long best_t = kClosest0;       // per-cell closest of MY ray
        unsigned best_tri = ~0u;
#endif
        __syncwarp();
        // (owner lane, list position) of item rbase + lane; rbase is warp-uniform and every lane takes part
        auto locate = [&](unsigned rbase, unsigned& owner, unsigned& pos) {
#if RM_TRAV_EXCL_SHARED
            const unsigned excl = sh.excl[lane];
#endif
            const unsigned first = __popc(__ballot_sync(FULL, excl <= rbase)) - 1u;
            const unsigned off = excl - rbase;                                   // 1..31 when my list starts inside the round
            const unsigned bits = __reduce_or_sync(FULL, (off - 1u < 31u) ? (1u << off) : 0u);
            const unsigned item = rbase + lane;
            if (item < total) {
                const unsigned q = first + __popc(bits & ((2u << lane) - 1u));
                owner = sh.olane[q];
                pos = item + sh.odelta[q];
            }
        };
        // Two stages, both with full lanes.  Stage 1: a round of 32 candidates is located, their bounding spheres and triangle
        // indices (16 B + 4 B, contiguous per cell: coalesced reads, fetched one round ahead) are read, the spheres tested, and
        // the candidates whose ray provably misses are dropped; survivors are appended (ballot compaction, order kept) to a ring
        // in shared memory and their 96-B records start towards L1.
        // Stage 2, whenever 32 survivors wait (or the pool is exhausted): 96-B record -> Triangle::intersects.
        unsigned owner = 0, pos = 0;
        float4 sp = make_float4(0.f, 0.f, 0.f, 0.f);
        locate(0u, owner, pos);
        if (lane < total) sp = __ldg(&g.sphr[pos]);
        unsigned tri = 0;                                    // ... and its triangle index (same index: one more coalesced read)
        if (lane < total) tri = __ldg(&g.refs[pos]);
        unsigned base = 0, q_head = 0, q_count = 0;          // warp-uniform
        for (;;) {
            if (base < total && q_count < 32u) {
                const bool valid = base + lane < total;
                const unsigned c_owner = owner;
                const float4 c_sp = sp;
                const unsigned c_tri1 = tri;
                if (base + 32u < total) {                    // warp-uniform
                    locate(base + 32u, owner, pos);
                    if (base + 32u + lane < total) {
                        sp = __ldg(&g.sphr[pos]);
                        tri = __ldg(&g.refs[pos]);
                    }
                }
                bool pass = false;
                if (valid) {
                    const double2 r0 = sh.ray[c_owner][0], r1 = sh.ray[c_owner][1], r2 = sh.ray[c_owner][2];
                    const double2 dl = sh.dd_lim[c_owner];
                    pass = !cull_sphere(c_sp, d3(r0.x, r0.y, r1.x), d3(r1.y, r2.x, r2.y), dl.x, dl.y);
                }
                const unsigned m = __ballot_sync(FULL, pass);
                if (pass) {
                    const unsigned slot = (q_head + q_count + __popc(m & lt)) & 63u;
                    sh.s_tri[slot] = c_tri1; sh.s_owner[slot] = (unsigned char)c_owner;
                    // the survivor's 96-B record (up to two lines) starts towards L1 now; stage 2 reads it a few rounds later
                    const double* tp = g.tri + (size_t)c_tri1 * 12;
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(tp));
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(tp + 8));
                }
                q_count += __popc(m);
                if (COUNT && pass) n_surv++;
                base += 32u;
                __syncwarp();
                RM_PROF_MARK(5);
                continue;
            }
            if (q_count == 0u) break;
            const unsigned take = q_count < 32u ? q_count : 32u;
            const bool valid = lane < take;
            bool got = false;
            unsigned long long tb = 0;
            unsigned c_owner = 0;
            const unsigned slot = (q_head + lane) & 63u;
            if (valid) {
                c_owner = sh.s_owner[slot];
                const TriPos tp = load_triangle(g.tri + (size_t)sh.s_tri[slot] * 12);
                const double2 r0 = sh.ray[c_owner][0], r1 = sh.ray[c_owner][1], r2 = sh.ray[c_owner][2];
                double t;
                unsigned fl = 0;
                const bool is_hit = hit_triangle(tp, d3(r0.x, r0.y, r1.x), d3(r1.y, r2.x, r2.y), t, COUNT ? &fl : nullptr);
                if (COUNT) n_flops += fl;
                if (is_hit) {
                    tb = (unsigned long long)__double_as_longlong(t);      // t > 1e-8: bit order = numeric order
                    got = true;
                    atomicMin(&sh.cand_t[c_owner], tb);
                }
            }
            q_head = (q_head + take) & 63u;
            q_count -= take;
            if (__any_sync(FULL, got)) {
                __syncwarp();
                if (got && sh.cand_t[c_owner] == tb) atomicMin(&sh.cand_tri[c_owner], sh.s_tri[slot]);   // (the ring slot is read again: hits are rare)
                __syncwarp();
                // strict < against the earlier rounds (they hold earlier list positions) and against 5712515.0
                const unsigned long long ct = sh.cand_t[lane];
#if RM_TRAV_PARK
                if (ct < sh.cell_t[lane]) { sh.cell_t[lane] = ct; sh.cell_tri[lane] = sh.cand_tri[lane]; }
#else
                if (ct < best_t) { best_t = ct; best_tri = sh.cand_tri[lane]; }
#endif
                sh.cand_t[lane] = ~0ull;
                sh.cand_tri[lane] = ~0u;
            }
            __syncwarp();       // the ring slots just read may be rewritten by the next stage-1 round
            RM_PROF_MARK(6);
        }
        RM_PROF_MARK(2);
        // ---- C
#if RM_TRAV_PARK
        state = sh.state[lane];
#endif
        if (state == TS_READY) {
#if RM_TRAV_PARK
            const unsigned best_tri = sh.cell_tri[lane];
            const unsigned long long best_t = sh.cell_t[lane];
#endif
            if (best_tri != ~0u) {
                const double closest = __longlong_as_double((long long)best_t);
                // the cell's closest hit is the grid's answer; merge with what the other objects found (the hit record of
                // this ray as k_setup left it came in with the traversal record: no global read here)
                if (closer(closest, a.grid_object, sh.best_t[lane], sh.best_obj[lane])) {
#if RM_TRAV_PARK
                    const unsigned ray = sh.ray_index[lane];
#endif
                    a.hit.t[ray] = closest; a.hit.obj[ray] = a.grid_object; a.hit.sub[ray] = best_tri;
                }
                state = TS_IDLE;
            } else {
                state = TS_STEP;
            }
        }
        __syncwarp();       // shared rays / prefix are rewritten by the next iteration
        RM_PROF_MARK(3);
    }
#if defined(RM_TRAV_PROFILE)
    if (lane == 0) {
        for (int i = 0; i < 7; i++) atomicAdd(&g_trav_prof[i], prof[i]);
        atomicAdd(&g_trav_prof[7], 1ull);
    }
#endif
    if (COUNT) {
        const unsigned c = __reduce_add_sync(FULL, n_cells), t = __reduce_add_sync(FULL, n_tests);
        const unsigned sv = __reduce_add_sync(FULL, n_surv), oc = __reduce_add_sync(FULL, n_occ), fl = __reduce_add_sync(FULL, n_flops);
        if (lane == 0) {
            atomicAdd(&a.totals->cells[stage_slot(a.depth)], (unsigned long long)c);
            atomicAdd(&a.totals->tests[stage_slot(a.depth)], (unsigned long long)t);
            atomicAdd(&a.totals->survivors[stage_slot(a.depth)], (unsigned long long)sv);
            atomicAdd(&a.totals->occupied[stage_slot(a.depth)], (unsigned long long)oc);
            atomicAdd(&a.totals->test_flops[stage_slot(a.depth)], (unsigned long long)fl);
        }
    }
}

// Stage part 3: shade, then deliver radiance or append the next ray (warp-aggregated compaction) to the next depth's queue.
// KEEP = RM_FLAG_KEEP_NONFINITE: the path's value is formed as the reference forms it, so that a NaN / Inf weight anywhere on
// the path poisons the sample: no path is stopped for a zero throughput (D5), and a path that ends without emission delivers
// T (*) 0 on a miss and T (*) w (*) 0 at the bounce limit instead of an exact (0, 0, 0).  The default instantiation is the
// one the benchmark runs.
// LAST (drop mode, depth == bounce_limit): shade() ends every path there, delivering T (*) emission for an emitter hit and an
// exact (0, 0, 0) otherwise, so this instantiation reads only the hit object, the slot and the throughput of emitter hits,
// and forms T (*) emission with the same multiplication as the general body.  No path continues and no triangle is shaded.
template <bool FIRST, int PREC, bool KEEP, bool LAST>
__global__ void __launch_bounds__(kBlock, RM_SHADE_BLOCKS_PER_SM) k_shade(const __grid_constant__ DevScene sc, const __grid_constant__ RenderParams rp, const Queue qin,
                                                   const Queue qout, const HitArrays hit, const unsigned depth, const unsigned n_first) {
    static_assert(!(LAST && KEEP), "keep mode computes the last weight: it has no last-depth shortcut");
    const unsigned n = FIRST ? n_first : rp.cnt.rays[depth - 1];
    const unsigned lane = threadIdx.x & 31u;
    const unsigned warps_total = (gridDim.x * blockDim.x) >> 5;
    const unsigned warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (LAST) {
        for (unsigned i = warp * 32u + lane; i < n; i += warps_total * 32u) {
            const unsigned slot = FIRST ? i : qin.id[i];
            const int ob = hit.obj[i];
            D3 result = d3(0.0, 0.0, 0.0);
            if (ob >= 0 && sc.obj[ob].mat == RM_MATERIAL_EMISSION)
                result = mul(FIRST ? d3(1.0, 1.0, 1.0) : d3(qin.f[6][i], qin.f[7][i], qin.f[8][i]), ld3(sc.obj[ob].color));
            rp.contrib[slot] = result.x;
            rp.contrib[(size_t)rp.cap + slot] = result.y;
            rp.contrib[2 * (size_t)rp.cap + slot] = result.z;
        }
        return;
    }
    unsigned shaded_tri = 0;
    for (unsigned base = warp * 32u; base < n; base += warps_total * 32u) {
        const unsigned i = base + lane;
        bool cont = false;
        D3 o, d, T;
        unsigned slot = 0;
        if (i < n) {
            slot = FIRST ? i : qin.id[i];
            o = d3(qin.f[0][i], qin.f[1][i], qin.f[2][i]);
            d = d3(qin.f[3][i], qin.f[4][i], qin.f[5][i]);
            const unsigned q = slot % rp.n_pixels, s_local = slot / rp.n_pixels;
            D3 v = d3(0.0, 0.0, 0.0);
            const Bounce b = shade<PREC, KEEP>(sc, rp, hit.t[i], hit.obj[i], hit.sub[i], rp.pixel_map[q], rp.first_sample + s_local * rp.sample_stride, depth, o, d, v, shaded_tri);
            // the path's value is (prod of weights) (*) emission (src/trace.rs:281-282,315-319): the throughput so far comes in only now
            T = d3(0.0, 0.0, 0.0);
            if (KEEP || b != BOUNCE_NONE) T = mul(FIRST ? d3(1.0, 1.0, 1.0) : d3(qin.f[6][i], qin.f[7][i], qin.f[8][i]), v);
            if (KEEP) cont = b == BOUNCE_CONTINUE;
            else cont = b == BOUNCE_CONTINUE && !(T.x == 0.0 && T.y == 0.0 && T.z == 0.0);   // nothing downstream can change a zero path value
            if (!cont) {
                const D3 result = b == BOUNCE_EMIT ? T : KEEP ? mul(T, d3(0.0, 0.0, 0.0)) : d3(0.0, 0.0, 0.0);
                rp.contrib[slot] = result.x;
                rp.contrib[(size_t)rp.cap + slot] = result.y;
                rp.contrib[2 * (size_t)rp.cap + slot] = result.z;
            }
        }
        const unsigned mask = __ballot_sync(0xffffffffu, cont);
        if (mask) {
            unsigned pos = 0;
            if (lane == 0) pos = atomicAdd(&rp.cnt.rays[depth], (unsigned)__popc(mask));
            pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(mask & ((1u << lane) - 1u));
            if (cont) {
                qout.id[pos] = slot;
                qout.f[0][pos] = o.x; qout.f[1][pos] = o.y; qout.f[2][pos] = o.z;
                qout.f[3][pos] = d.x; qout.f[4][pos] = d.y; qout.f[5][pos] = d.z;
                qout.f[6][pos] = T.x; qout.f[7][pos] = T.y; qout.f[8][pos] = T.z;
            }
        }
    }
    shaded_tri = __reduce_add_sync(0xffffffffu, shaded_tri);
    if (lane == 0 && shaded_tri) atomicAdd(&rp.totals->shaded[stage_slot(depth)], (unsigned long long)shaded_tri);
}

// tile.data[..] += sample, one pass after the other          src/trace.rs:203
// Adds the batch's per-path radiance to the running sums in global sample order, so the
// association is the reference's ((0 + s0) + s1) + ...  Non-finite samples are dropped and counted
// unless RM_FLAG_KEEP_NONFINITE.  MOMENTS (RM_FLAG_MOMENTS): the same samples' squares go into `moments`, in the same order.
// `moments` is the last parameter so that the default instantiation keeps the parameter layout (and the code) it always had.
template <bool MOMENTS>
__global__ void __launch_bounds__(kBlock) k_accumulate(const __grid_constant__ RenderParams rp, double* __restrict__ accum,
                                                        const unsigned n_batch_samples, const unsigned keep_nonfinite, double* __restrict__ moments) {
    DevTotals* totals = rp.totals;
    const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned bad = 0;
    if (q < rp.n_pixels) {
        const size_t p = (size_t)rp.pixel_map[q] * 3;
        double sx = accum[p], sy = accum[p + 1], sz = accum[p + 2];
        double qx = 0.0, qy = 0.0, qz = 0.0;
        if (MOMENTS) { qx = moments[p]; qy = moments[p + 1]; qz = moments[p + 2]; }
        for (unsigned s = 0; s < n_batch_samples; s++) {
            const size_t k = (size_t)s * rp.n_pixels + q;
            const double cx = rp.contrib[k], cy = rp.contrib[(size_t)rp.cap + k], cz = rp.contrib[2 * (size_t)rp.cap + k];
            const bool finite = isfinite(cx) && isfinite(cy) && isfinite(cz);
            if (!finite) bad++;
            if (finite || keep_nonfinite) {
                sx += cx; sy += cy; sz += cz;
                if (MOMENTS) { qx += cx * cx; qy += cy * cy; qz += cz * cz; }
            }
        }
        accum[p] = sx; accum[p + 1] = sy; accum[p + 2] = sz;
        if (MOMENTS) { moments[p] = qx; moments[p + 1] = qy; moments[p + 2] = qz; }
    }
    bad = __reduce_add_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31u) == 0 && bad) atomicAdd(&totals->nonfinite, (unsigned long long)bad);
    if (q == 0) {
        unsigned long long rays = (unsigned long long)n_batch_samples * rp.n_pixels;
        if (rp.bounce_limit) totals->stage_rays[1] += rays;
        for (unsigned dpt = 1; dpt < rp.bounce_limit; dpt++) { rays += rp.cnt.rays[dpt]; totals->stage_rays[stage_slot(dpt + 1)] += rp.cnt.rays[dpt]; }
        totals->rays += rp.bounce_limit ? rays : 0ull;
        totals->samples += (unsigned long long)n_batch_samples * rp.n_pixels;
    }
}

// Sums of several renderers' accumulators (and second moments), read in place in device order like the accumulator exchange.
constexpr int kMaxShares = 64;
struct ShareMoments {
    const double* acc[kMaxShares];
    const double* mom[kMaxShares];
    int count;
};

// E_t of one tile per block (include/raymond.h, rm_adaptive_settings): tile `first + blockIdx.x * step` of the layout, the
// tiles in the reference's column-major order.  Every thread sums r_p^2 over a fixed stride of the tile's pixels, then a fixed
// tree in shared memory: the result does not depend on scheduling.  max(x, 0) keeps a NaN (a NaN tile never converges).
constexpr int kTileErrorBlock = 256;
__global__ void __launch_bounds__(kTileErrorBlock) k_tile_error(const __grid_constant__ ShareMoments sm, double* __restrict__ out, unsigned W, unsigned H,
                                                                 unsigned tw, unsigned th, unsigned first, unsigned step, double n) {
    __shared__ double part[kTileErrorBlock];
    const unsigned t = first + blockIdx.x * step;
    const unsigned tiles_y = (H + th - 1) / th;
    const unsigned left = (t / tiles_y) * tw, top = (t % tiles_y) * th;
    const unsigned w = min(tw, W - left), h = min(th, H - top);
    double acc = 0.0;
    for (unsigned k = threadIdx.x; k < w * h; k += kTileErrorBlock) {
        const size_t p = ((size_t)(top + k / w) * W + left + k % w) * 3;
        double se2 = 0.0, msum = 0.0;
        for (int c = 0; c < 3; c++) {
            double S = sm.acc[0][p + c], Q = sm.mom[0][p + c];
            for (int j = 1; j < sm.count; j++) { S += sm.acc[j][p + c]; Q += sm.mom[j][p + c]; }
            const double m = S / n;
            const double d = Q - S * m;
            const double v = (d < 0.0 ? 0.0 : d) / (n - 1.0);
            se2 += v / n;
            msum += m;
        }
        const double r = sqrt(se2) / (msum + 1e-3);
        acc += r * r;
    }
    part[threadIdx.x] = acc;
    __syncthreads();
    for (unsigned half = kTileErrorBlock / 2; half > 0; half >>= 1) {
        if (threadIdx.x < half) part[threadIdx.x] += part[threadIdx.x + half];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[t] = sqrt(part[0] / (double)(w * h));
}

// Active-tile compaction: entry i = {source offset, destination offset, length} copies one tile's run of the full pixel map.
__global__ void __launch_bounds__(kBlock) k_gather_pixels(const unsigned* __restrict__ src, const uint3* __restrict__ runs, unsigned* __restrict__ dst) {
    const uint3 e = runs[blockIdx.x];
    for (unsigned k = threadIdx.x; k < e.z; k += blockDim.x) dst[e.y + k] = src[e.x + k];
}

// Hit records -> the caller's Scene::intersect outputs (distance left untouched on a miss).
__global__ void __launch_bounds__(kBlock) k_export_hits(const HitArrays hit, const size_t n, long long* __restrict__ obj,
                                                         unsigned long long* __restrict__ sub, double* __restrict__ dist_out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int ob = hit.obj[i];
        if (obj) obj[i] = ob;
        if (sub) sub[i] = ob >= 0 ? hit.sub[i] : 0ull;
        if (dist_out && ob >= 0) dist_out[i] = hit.t[i];
    }
}

// generate_primary_ray with the jitter term forced to 0, whole frame, row-major.
__global__ void __launch_bounds__(kBlock) k_primary_rays(const __grid_constant__ DevCamera cam, rm_ray* __restrict__ rays) {
    const size_t n = (size_t)cam.W * cam.H;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const D3 d = primary_direction(cam, (unsigned)(i % cam.W), (unsigned)(i / cam.W), 0.0, 0.0);
        double* r = reinterpret_cast<double*>(rays + i);
        r[0] = cam.pos[0]; r[1] = cam.pos[1]; r[2] = cam.pos[2];
        r[3] = d.x; r[4] = d.y; r[5] = d.z;
    }
}

}  // namespace rm
