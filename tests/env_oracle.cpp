// env_oracle.cpp — the CPU oracle with an environment map (test infrastructure only; built by tests/env_oracle.py).
//
// The reference's Scene has no environment, so the oracle (oracle/raymond_oracle.cpp) has none either and stays as it is.
// This file includes it unchanged and adds, next to it:
//   env_radiance   the lookup of include/raymond.h (rm_environment) with glibc's atan2 / acos, f64, in the header's order;
//   trace_env      `trace` (src/trace.rs:232-320) with one change: a ray that misses every object at depth <= bounce_limit
//                  returns env_radiance(direction) instead of 0 — the product's semantics with a map;
//   rmoe_*         a C API over them: the lookup alone, and one sample per pixel of a frame (like rmo_render with
//                  sample_count 1, first_sample = sample).
// Build: g++ -O2 -std=c++17 -fPIC -ffp-contract=off -shared -pthread (the oracle's flags).
#include "../oracle/raymond_oracle.cpp"

namespace {

struct Environment { std::vector<float> texels; size_t width = 0, height = 0; double scale = 1.0, rotation = 0.0; };

V3 env_radiance(const Environment& e, V3 d) {
    double u = 0.5 + (std::atan2(d.x, d.z) + e.rotation) / (2.0 * PI);
    u -= std::floor(u);
    const double cy = d.y < -1.0 ? -1.0 : d.y > 1.0 ? 1.0 : d.y;
    const double v = std::acos(cy) / PI;
    if (std::isnan(u) || std::isnan(v)) { const double nan = std::nan(""); return v3(nan, nan, nan); }
    const double x = u * (double)e.width - 0.5, y = v * (double)e.height - 0.5;
    const double x0 = std::floor(x), y0 = std::floor(y);
    const double fx = x - x0, fy = y - y0;
    const long W = (long)e.width, H = (long)e.height;
    long ix0 = (long)x0, iy0 = (long)y0, ix1 = ix0 + 1, iy1 = iy0 + 1;
    ix0 = ((ix0 % W) + W) % W; ix1 = ((ix1 % W) + W) % W;
    iy0 = std::min(std::max(iy0, 0L), H - 1); iy1 = std::min(std::max(iy1, 0L), H - 1);
    auto t = [&](long r, long c) { const float* p = &e.texels[3 * (size_t)(r * W + c)]; return v3(p[0], p[1], p[2]); };
    const V3 top = t(iy0, ix0) + fx * (t(iy0, ix1) - t(iy0, ix0));
    const V3 bot = t(iy1, ix0) + fx * (t(iy1, ix1) - t(iy1, ix0));
    return e.scale * (top + fy * (bot - top));
}

// `trace` of raymond_oracle.cpp, statement for statement, except on a miss
V3 trace_env(const Ray& ray, const TraceContext& ctx, const Environment& env, size_t depth, const Sampler& rng) {
    const Settings& settings = *ctx.settings;
    if (depth > settings.bounce_limit) return v3(0.0, 0.0, 0.0);

    size_t oi; Hit hit;
    if (!scene_intersect(*ctx.scene, ray, &oi, &hit)) return env_radiance(env, ray.direction);      // the one change
    const Object& object = ctx.scene->objects[oi];
    V3 normal = surface_normal(object, ray, hit);
    V3 fragment_position = ray.origin + ray.direction * hit.distance;
    V3 material_color; double material_roughness, material_metalness;
    switch (object.material.kind) {
        case MAT_DIFFUSE: material_color = object.material.a; material_roughness = object.material.p0; material_metalness = 0.0; break;
        case MAT_METAL: material_color = object.material.a; material_roughness = object.material.p0; material_metalness = 1.0; break;
        default: return object.material.a;
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
        V3 radiance = trace_env(Ray{fragment_position + normal * 0.00001, sample_world}, ctx, env, depth + 1, rng);
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
        V3 radiance = trace_env(Ray{fragment_position + normal * 0.0001, sample_world}, ctx, env, depth + 1, rng);
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

struct rmoe_env { Environment e; };

rmoe_env* rmoe_env_create(const float* texels, size_t width, size_t height, double scale, double rotation) {
    rmoe_env* h = new rmoe_env();
    h->e.texels.assign(texels, texels + 3 * width * height);
    h->e.width = width; h->e.height = height; h->e.scale = scale; h->e.rotation = rotation;
    return h;
}
void rmoe_env_destroy(rmoe_env* h) { delete h; }

// L(d) for n directions (n x 3) into out (n x 3)
void rmoe_env_lookup(const rmoe_env* h, const double* dirs, size_t n, double* out) {
    for (size_t i = 0; i < n; i++) {
        const V3 L = env_radiance(h->e, v3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]));
        out[3 * i] = L.x; out[3 * i + 1] = L.y; out[3 * i + 2] = L.z;
    }
}

// One sample of every pixel: out[p] = trace_env(camera_ray(p)) of global sample `sample` (W*H*3, row-major; zeros where a
// non-finite sample is dropped).  flags as rmo_render's: bit 0 drops (and counts) non-finite samples, bit 1 the f32-draw stream.
int rmoe_render_sample(const rmo_scene* scene, const rmoe_env* env, const rmo_settings* s, uint64_t seed, uint32_t sample,
                       uint32_t flags, int threads, double* out, rmo_counters* counters) {
    Settings settings = tosettings(*s);
    const size_t W = settings.camera_settings.backbuffer_width, H = settings.camera_settings.backbuffer_height;
    TraceContext ctx{&scene->s, &settings};
    if (threads < 1) threads = 1;
    std::vector<Counters> per((size_t)threads);
    auto work = [&](int k) {
        tl_counters = Counters{};
        for (size_t y = (size_t)k; y < H; y += (size_t)threads)
            for (size_t x = 0; x < W; x++) {
                Sampler rng{seed, (uint32_t)(x + y * W), sample, (flags & 2u) != 0};
                V3 smp = trace_env(camera_ray(x, y, settings.camera_settings, rng), ctx, env->e, 1, rng);
                tl_counters.samples++;
                const bool finite = std::isfinite(smp.x) && std::isfinite(smp.y) && std::isfinite(smp.z);
                if (!finite) { tl_counters.nonfinite++; if (flags & 1u) smp = v3(0.0, 0.0, 0.0); }
                double* o = out + 3 * (x + y * W);
                o[0] = 0.0 + smp.x; o[1] = 0.0 + smp.y; o[2] = 0.0 + smp.z;     // the running sum of one sample, as rmo_render keeps it
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
