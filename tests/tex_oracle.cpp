// tex_oracle.cpp — the CPU oracle with colour textures (test infrastructure only; built by tests/tex_oracle.py).
//
// The reference's materials have one colour, so the oracle (oracle/raymond_oracle.cpp) has no textures and stays as it is.
// This file includes tests/env_oracle.cpp (the oracle and its environment map) unchanged and adds, next to it:
//   tex_lookup     T(s, t) of include/raymond.h (rm_texture), f64, in the header's order;
//   hit_uv         the (s, t) of a hit on a plane, a sphere (glibc's atan2 / acos) or a grid triangle;
//   trace_tex      trace_env statement for statement, with material_color = a (*) T(s, t) for a textured object;
//   rmot_*         a C API over them: the lookup, the uv of each geometry kind, and one sample per pixel of a frame.
// Build: g++ -O2 -std=c++17 -fPIC -ffp-contract=off -shared -pthread (the oracle's flags).
#include "env_oracle.cpp"

namespace {

struct Texture { std::vector<float> texels; size_t width = 0, height = 0; double su = 1.0, sv = 1.0; };

V3 tex_lookup(const Texture& x, double s, double t) {
    double sp = s * x.su, tp = t * x.sv;
    if (!std::isfinite(sp) || !std::isfinite(tp)) { const double nan = std::nan(""); return v3(nan, nan, nan); }
    sp -= std::floor(sp);
    tp -= std::floor(tp);
    const double fxx = sp * (double)x.width - 0.5, fyy = (1.0 - tp) * (double)x.height - 0.5;
    const double x0 = std::floor(fxx), y0 = std::floor(fyy);
    const double fx = fxx - x0, fy = fyy - y0;
    const long W = (long)x.width, H = (long)x.height;
    long ix0 = (long)x0, iy0 = (long)y0, ix1 = ix0 + 1, iy1 = iy0 + 1;
    ix0 = ((ix0 % W) + W) % W; ix1 = ((ix1 % W) + W) % W;
    iy0 = ((iy0 % H) + H) % H; iy1 = ((iy1 % H) + H) % H;
    auto t_ = [&](long r, long c) { const float* p = &x.texels[3 * (size_t)(r * W + c)]; return v3(p[0], p[1], p[2]); };
    const V3 top = t_(iy0, ix0) + fx * (t_(iy0, ix1) - t_(iy0, ix0));
    const V3 bot = t_(iy1, ix0) + fx * (t_(iy1, ix1) - t_(iy1, ix0));
    return top + fy * (bot - top);
}

V2 sphere_uv(V3 n) {
    const double s = 0.5 + std::atan2(n.x, n.z) / (2.0 * PI);
    const double cy = n.y < -1.0 ? -1.0 : n.y > 1.0 ? 1.0 : n.y;
    return V2{s, 1.0 - std::acos(cy) / PI};
}

V2 plane_uv(V3 origin, V3 normal, V3 frag) {
    V3 tg, bt;
    create_coordinate_system_of_n(normal, &tg, &bt);
    const V3 p = frag - origin;
    return V2{dot(p, tg), dot(p, bt)};
}

// the Heron weights of triangle_normal (triangle.rs:47-68), then the normal's own expression on the vertices' uv
V2 triangle_uv(const Triangle& tri, V3 position) {
    double abc = heron_area(tri.v0.position, tri.v1.position, tri.v2.position);
    double abp = heron_area(tri.v0.position, tri.v1.position, position);
    double bcp = heron_area(tri.v0.position, tri.v2.position, position);
    double ba = abp / abc;
    double bb = bcp / abc;
    double bc = 1.0 - (ba + bb);
    return V2{((tri.v2.uv.x * ba) + (tri.v1.uv.x * bb)) + (tri.v0.uv.x * bc), ((tri.v2.uv.y * ba) + (tri.v1.uv.y * bb)) + (tri.v0.uv.y * bc)};
}

V2 hit_uv(const Object& o, V3 normal, V3 frag, const Hit& hit) {
    switch (o.geometry) {
        case GEO_PLANE: return plane_uv(o.origin, o.normal, frag);
        case GEO_SPHERE: return sphere_uv(normal);
        default: return triangle_uv(o.grid->mesh.triangles[hit.subobject_index], frag);
    }
}

// per object: its texture or null
using Textures = std::vector<const Texture*>;

// `trace_env` of env_oracle.cpp, statement for statement, except for the colour of a textured object
V3 trace_tex(const Ray& ray, const TraceContext& ctx, const Environment& env, const Textures& tex, size_t depth, const Sampler& rng) {
    const Settings& settings = *ctx.settings;
    if (depth > settings.bounce_limit) return v3(0.0, 0.0, 0.0);

    size_t oi; Hit hit;
    if (!scene_intersect(*ctx.scene, ray, &oi, &hit)) return env_radiance(env, ray.direction);
    const Object& object = ctx.scene->objects[oi];
    V3 normal = surface_normal(object, ray, hit);
    V3 fragment_position = ray.origin + ray.direction * hit.distance;
    V3 material_color; double material_roughness, material_metalness;
    switch (object.material.kind) {
        case MAT_DIFFUSE: material_color = object.material.a; material_roughness = object.material.p0; material_metalness = 0.0; break;
        case MAT_METAL: material_color = object.material.a; material_roughness = object.material.p0; material_metalness = 1.0; break;
        default: return object.material.a;
    }
    if (oi < tex.size() && tex[oi]) {                                                                   // the one change
        const V2 uv = hit_uv(object, normal, fragment_position, hit);
        material_color = mul_ew(material_color, tex_lookup(*tex[oi], uv.x, uv.y));
    }

    V3 view_dir = normalize(settings.camera_settings.position - fragment_position);
    V3 f0 = v3(0.04, 0.04, 0.04);
    f0 = lerp_vec(f0, material_color, material_metalness);
    double r = rng.draw((uint32_t)depth, 0);
    V3 lc0, lc1;
    create_coordinate_system_of_n(normal, &lc0, &lc1);
    double prob_d = lerp(0.5, 0.0, material_metalness);
    if (r < prob_d) {
        V3 sample; double pdf;
        uniform_sample_hemisphere(rng.draw((uint32_t)depth, 1), rng.draw((uint32_t)depth, 2), &sample, &pdf);
        V3 sample_world = normalize(mat_mul(lc0, normal, lc1, sample));
        V3 radiance = trace_tex(Ray{fragment_position + normal * 0.00001, sample_world}, ctx, env, tex, depth + 1, rng);
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
        V3 radiance = trace_tex(Ray{fragment_position + normal * 0.0001, sample_world}, ctx, env, tex, depth + 1, rng);
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

}  // namespace

extern "C" {

struct rmot_tex { Texture t; };

rmot_tex* rmot_tex_create(const float* texels, size_t width, size_t height, double su, double sv) {
    rmot_tex* h = new rmot_tex();
    h->t.texels.assign(texels, texels + 3 * width * height);
    h->t.width = width; h->t.height = height; h->t.su = su; h->t.sv = sv;
    return h;
}
void rmot_tex_destroy(rmot_tex* h) { delete h; }

// T(s, t) for n uv pairs (n x 2) into out (n x 3)
void rmot_tex_lookup(const rmot_tex* h, const double* st, size_t n, double* out) {
    for (size_t i = 0; i < n; i++) {
        const V3 T = tex_lookup(h->t, st[2 * i], st[2 * i + 1]);
        out[3 * i] = T.x; out[3 * i + 1] = T.y; out[3 * i + 2] = T.z;
    }
}

// (s, t) of n sphere normals (n x 3)
void rmot_sphere_uv(const double* normals, size_t n, double* out) {
    for (size_t i = 0; i < n; i++) {
        const V2 uv = sphere_uv(v3(normals[3 * i], normals[3 * i + 1], normals[3 * i + 2]));
        out[2 * i] = uv.x; out[2 * i + 1] = uv.y;
    }
}

// (s, t) of n hit points on the plane (origin, normal)
void rmot_plane_uv(const double* origin, const double* normal, const double* frags, size_t n, double* out) {
    for (size_t i = 0; i < n; i++) {
        const V2 uv = plane_uv(v3(origin[0], origin[1], origin[2]), v3(normal[0], normal[1], normal[2]), v3(frags[3 * i], frags[3 * i + 1], frags[3 * i + 2]));
        out[2 * i] = uv.x; out[2 * i + 1] = uv.y;
    }
}

// (s, t) of n hit points, point i on reference-layout triangle i (264 bytes each)
void rmot_triangle_uv(const void* tris, const double* points, size_t n, double* out) {
    for (size_t i = 0; i < n; i++) {
        Triangle t;
        std::memcpy(&t, (const char*)tris + i * sizeof(Triangle), sizeof(Triangle));
        const V2 uv = triangle_uv(t, v3(points[3 * i], points[3 * i + 1], points[3 * i + 2]));
        out[2 * i] = uv.x; out[2 * i + 1] = uv.y;
    }
}

// One sample of every pixel with the textures `tex` (one handle or null per object; n_tex entries): as rmoe_render_sample.
int rmot_render_sample(const rmo_scene* scene, const rmoe_env* env, const rmot_tex* const* tex, size_t n_tex, const rmo_settings* s, uint64_t seed,
                       uint32_t sample, uint32_t flags, int threads, double* out, rmo_counters* counters) {
    Settings settings = tosettings(*s);
    const size_t W = settings.camera_settings.backbuffer_width, H = settings.camera_settings.backbuffer_height;
    TraceContext ctx{&scene->s, &settings};
    Textures textures(n_tex, nullptr);
    for (size_t i = 0; i < n_tex; i++) textures[i] = tex[i] ? &tex[i]->t : nullptr;
    if (threads < 1) threads = 1;
    std::vector<Counters> per((size_t)threads);
    auto work = [&](int k) {
        tl_counters = Counters{};
        for (size_t y = (size_t)k; y < H; y += (size_t)threads)
            for (size_t x = 0; x < W; x++) {
                Sampler rng{seed, (uint32_t)(x + y * W), sample, (flags & 2u) != 0};
                V3 smp = trace_tex(camera_ray(x, y, settings.camera_settings, rng), ctx, env->e, textures, 1, rng);
                tl_counters.samples++;
                const bool finite = std::isfinite(smp.x) && std::isfinite(smp.y) && std::isfinite(smp.z);
                if (!finite) { tl_counters.nonfinite++; if (flags & 1u) smp = v3(0.0, 0.0, 0.0); }
                double* o = out + 3 * (x + y * W);
                o[0] = 0.0 + smp.x; o[1] = 0.0 + smp.y; o[2] = 0.0 + smp.z;
            }
        per[(size_t)k] = tl_counters;
    };
    std::vector<std::thread> th;
    for (int k = 1; k < threads; k++) th.emplace_back(work, k);
    work(0);
    for (auto& t : th) t.join();
    Counters total; for (auto& c : per) total.add(c);
    export_counters(total, counters);
    return 0;
}

}  // extern "C"
